#!/usr/bin/env python3
"""Synthetic Pocket-TTS model directory in the REAL file layout (no network here).

Emits what `ptts_init` / `ptts_stream_from_safetensors` of the reference expect to find
under `model_path` (reference src/pocket_tts.cpp:241-250,292-293, src/config.h:71):

    <dir>/tts_b6369a24.safetensors      seeded random weights, real key names/shapes
    <dir>/tokenizer.model               SentencePiece unigram proto (copied from tests/golden)
    <dir>/embeddings/<voice>.safetensors   tensor "audio_prompt" [1, T_voice, 1024]

Key names = the names the reference fetches minus their first component
(src/loader.h:101-105), shapes are torch-order (SURVEY.md Appendix B).

The safetensors container is written by hand (8-byte LE header length, JSON header,
raw little-endian tensor bytes) so that BF16 needs neither torch nor ml_dtypes.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import struct
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
GOLDEN_TOKENIZER = os.path.join(REPO, "tests", "golden", "tokenizer.model")

VOICES = ["alba", "azelma", "cosette", "eponine", "fantine", "javert", "jean", "marius"]


# ----------------------------------------------------------------------------------
# dtype helpers
# ----------------------------------------------------------------------------------
def f32_to_bf16_bits(x: np.ndarray) -> np.ndarray:
    """Round-to-nearest-even fp32 -> bf16 bit pattern (uint16)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    rounding = ((u >> 16) & 1) + 0x7FFF
    return ((u + rounding) >> 16).astype(np.uint16)


def bf16_bits_to_f32(b: np.ndarray) -> np.ndarray:
    return (b.astype(np.uint32) << 16).view(np.float32)


def write_safetensors(path: str, tensors: dict[str, np.ndarray], dtype: str) -> None:
    """tensors: name -> float32 ndarray. dtype: 'BF16' | 'F32' (file dtype of every tensor)."""
    header = {}
    blobs = []
    off = 0
    for name, arr in tensors.items():
        arr = np.ascontiguousarray(arr, dtype=np.float32)
        if dtype == "BF16":
            raw = f32_to_bf16_bits(arr).tobytes()
        elif dtype == "F32":
            raw = arr.tobytes()
        else:
            raise ValueError(dtype)
        header[name] = {"dtype": dtype, "shape": list(arr.shape), "data_offsets": [off, off + len(raw)]}
        blobs.append(raw)
        off += len(raw)
    hjson = json.dumps(header, separators=(",", ":")).encode()
    pad = (8 - len(hjson) % 8) % 8
    hjson += b" " * pad
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(struct.pack("<Q", len(hjson)))
        f.write(hjson)
        for b in blobs:
            f.write(b)
    os.replace(tmp, path)


def read_safetensors(path: str) -> dict[str, np.ndarray]:
    """Reads F32/BF16/F16 tensors back as float32 (used by tests and the torch second opinion)."""
    with open(path, "rb") as f:
        (n,) = struct.unpack("<Q", f.read(8))
        header = json.loads(f.read(n))
        base = 8 + n
        out = {}
        for name, meta in header.items():
            if name == "__metadata__":
                continue
            a, b = meta["data_offsets"]
            f.seek(base + a)
            raw = f.read(b - a)
            if meta["dtype"] == "BF16":
                arr = bf16_bits_to_f32(np.frombuffer(raw, dtype=np.uint16))
            elif meta["dtype"] == "F32":
                arr = np.frombuffer(raw, dtype=np.float32)
            elif meta["dtype"] == "F16":
                arr = np.frombuffer(raw, dtype=np.float16).astype(np.float32)
            else:
                raise ValueError(meta["dtype"])
            out[name] = arr.reshape(meta["shape"]).copy()
        return out


# ----------------------------------------------------------------------------------
# weights
# ----------------------------------------------------------------------------------
def synth_weights(seed: int, eos_mode: str) -> dict[str, np.ndarray]:
    """Seeded random weights in the real key layout (SURVEY.md Appendix B / §8d)."""
    rng = np.random.default_rng(seed)
    W: dict[str, np.ndarray] = {}

    def lin(name, out_f, in_f, bias=False, gain=1.0):
        W[name + ".weight"] = (rng.standard_normal((out_f, in_f)) * (gain / np.sqrt(in_f))).astype(np.float32)
        if bias:
            W[name + ".bias"] = (rng.standard_normal(out_f) * 0.02).astype(np.float32)

    def norm(name, d):
        W[name + ".weight"] = (1.0 + 0.02 * rng.standard_normal(d)).astype(np.float32)
        W[name + ".bias"] = (0.02 * rng.standard_normal(d)).astype(np.float32)

    # ---- FlowLM (reference models/flow_lm.h:40-52, modules/transformer.h:16-19,215-225)
    W["flow_lm.conditioner.embed.weight"] = rng.standard_normal((4001, 1024)).astype(np.float32)
    W["flow_lm.emb_std"] = (1.0 + 0.1 * rng.random(32)).astype(np.float32)
    W["flow_lm.emb_mean"] = (0.1 * rng.standard_normal(32)).astype(np.float32)
    W["flow_lm.bos_emb"] = rng.standard_normal(32).astype(np.float32)
    lin("flow_lm.input_linear", 1024, 32)
    norm("flow_lm.out_norm", 1024)
    W["flow_lm.out_eos.weight"] = (rng.standard_normal((1, 1024)) / np.sqrt(1024)).astype(np.float32)
    if eos_mode == "never":
        # throughput checkpoints: logit ~ N(-10,1) never crosses the -4 threshold
        W["flow_lm.out_eos.bias"] = np.array([-10.0], dtype=np.float32)
    elif eos_mode == "mid":
        # parity checkpoints: P(logit_raw > 1.64) ~ 5 % per frame -> EOS lands mid-sentence
        W["flow_lm.out_eos.bias"] = np.array([-5.64], dtype=np.float32)
    elif eos_mode == "late":
        # ragged-throughput checkpoints: the raw logit has std ~1.2 over a generation (measured: bias -6.46 ended sentences after ~50 frames),
        # so -7.0 gives P(EOS) ~ 0.6 % per frame: sentences end after ~100+ frames or at their cap, i.e. raggedly
        W["flow_lm.out_eos.bias"] = np.array([-7.0], dtype=np.float32)
    else:
        raise ValueError(eos_mode)
    for l in range(6):
        p = f"flow_lm.transformer.layers.{l}."
        lin(p + "self_attn.in_proj", 3072, 1024)
        lin(p + "self_attn.out_proj", 1024, 1024, gain=0.5)
        norm(p + "norm1", 1024)
        norm(p + "norm2", 1024)
        lin(p + "linear1", 4096, 1024)
        lin(p + "linear2", 1024, 4096, gain=0.5)

    # ---- flow head (reference modules/mlp.h:80-87,117-122,150-154,221-231)
    f = "flow_lm.flow_net."
    lin(f + "input_proj", 512, 32, bias=True)
    lin(f + "cond_embed", 512, 1024, bias=True)
    for i in range(2):
        lin(f + f"time_embed.{i}.mlp.0", 512, 256, bias=True)
        lin(f + f"time_embed.{i}.mlp.2", 512, 512, bias=True)
        W[f + f"time_embed.{i}.mlp.3.alpha"] = (1.0 + 0.02 * rng.standard_normal(512)).astype(np.float32)
        W[f + f"time_embed.{i}.freqs"] = np.exp(-np.log(10000.0) * np.arange(128) / 128.0).astype(np.float32)
    for r in range(6):
        p = f + f"res_blocks.{r}."
        norm(p + "in_ln", 512)
        lin(p + "mlp.0", 512, 512, bias=True)
        lin(p + "mlp.2", 512, 512, bias=True)
        lin(p + "adaLN_modulation.1", 1536, 512, bias=True, gain=0.5)
    lin(f + "final_layer.linear", 32, 512, bias=True)
    lin(f + "final_layer.adaLN_modulation.1", 1024, 512, bias=True, gain=0.5)
    # final_layer.norm_final.* is optional in the reference (mlp.h:66-69) and absent here.

    # ---- Mimi (reference models/mimi.h:31-41, modules/mimi_transformer.h, modules/seanet.h:213-222)
    W["mimi.quantizer.output_proj.weight"] = (rng.standard_normal((512, 32, 1)) / np.sqrt(32)).astype(np.float32)
    W["mimi.upsample.convtr.convtr.weight"] = (rng.standard_normal((512, 1, 32)) * 0.7).astype(np.float32)
    for l in range(2):
        p = f"mimi.decoder_transformer.transformer.layers.{l}."
        norm(p + "norm1", 512)
        norm(p + "norm2", 512)
        lin(p + "self_attn.in_proj", 1536, 512)
        lin(p + "self_attn.out_proj", 512, 512)
        W[p + "layer_scale_1.scale"] = (0.1 + 0.01 * rng.standard_normal(512)).astype(np.float32)
        W[p + "layer_scale_2.scale"] = (0.1 + 0.01 * rng.standard_normal(512)).astype(np.float32)
        lin(p + "linear1", 2048, 512)
        lin(p + "linear2", 512, 2048)

    def conv(name, co, ci, k):
        W[name + ".conv.weight"] = (rng.standard_normal((co, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
        W[name + ".conv.bias"] = (0.02 * rng.standard_normal(co)).astype(np.float32)

    def convtr(name, ci, co, k, s):
        W[name + ".convtr.weight"] = (rng.standard_normal((ci, co, k)) / np.sqrt(ci * k / s)).astype(np.float32)
        W[name + ".convtr.bias"] = (0.02 * rng.standard_normal(co)).astype(np.float32)

    d = "mimi.decoder.model."
    conv(d + "0", 512, 512, 7)
    convtr(d + "2", 512, 256, 12, 6)
    conv(d + "3.block.1", 128, 256, 3)
    conv(d + "3.block.3", 256, 128, 1)
    convtr(d + "5", 256, 128, 10, 5)
    conv(d + "6.block.1", 64, 128, 3)
    conv(d + "6.block.3", 128, 64, 1)
    convtr(d + "8", 128, 64, 8, 4)
    conv(d + "9.block.1", 32, 64, 3)
    conv(d + "9.block.3", 64, 32, 1)
    conv(d + "11", 1, 64, 3)
    return W


def synth_encoder_weights(seed: int) -> dict[str, np.ndarray]:
    """The voice-cloning encoder set (DESIGN.md §4.6), drawn from its own generator so that the decoder-side stream is unchanged."""
    rng = np.random.default_rng([seed, 0xE1C])
    W: dict[str, np.ndarray] = {}

    def conv(name, co, ci, k, bias=True):
        W[name + ".conv.weight"] = (rng.standard_normal((co, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
        if bias:
            W[name + ".conv.bias"] = (0.02 * rng.standard_normal(co)).astype(np.float32)

    e = "mimi.encoder.model."
    conv(e + "0", 64, 1, 7)
    for i, c in ((1, 64), (4, 128), (7, 256)):
        conv(e + f"{i}.block.1", c // 2, c, 3)
        conv(e + f"{i}.block.3", c, c // 2, 1)
    conv(e + "3", 128, 64, 8)
    conv(e + "6", 256, 128, 10)
    conv(e + "9", 512, 256, 12)
    conv(e + "11", 512, 512, 3)
    for l in range(2):
        p = f"mimi.encoder_transformer.transformer.layers.{l}."
        for n in ("norm1", "norm2"):
            W[p + n + ".weight"] = (1.0 + 0.02 * rng.standard_normal(512)).astype(np.float32)
            W[p + n + ".bias"] = (0.02 * rng.standard_normal(512)).astype(np.float32)
        for n, o, i in (("self_attn.in_proj", 1536, 512), ("self_attn.out_proj", 512, 512), ("linear1", 2048, 512), ("linear2", 512, 2048)):
            W[p + n + ".weight"] = (rng.standard_normal((o, i)) / np.sqrt(i)).astype(np.float32)
        W[p + "layer_scale_1.scale"] = (0.1 + 0.01 * rng.standard_normal(512)).astype(np.float32)
        W[p + "layer_scale_2.scale"] = (0.1 + 0.01 * rng.standard_normal(512)).astype(np.float32)
    conv("mimi.downsample.conv", 512, 512, 32, bias=False)
    W["flow_lm.speaker_proj_weight"] = (rng.standard_normal((1024, 512)) / np.sqrt(512)).astype(np.float32)
    return W


def synth_voice(name: str, seed: int, t_voice: int) -> np.ndarray:
    h = sum((i + 1) * ord(c) for i, c in enumerate(name))
    rng = np.random.default_rng(seed * 1000003 + h)
    return rng.standard_normal((1, t_voice, 1024)).astype(np.float32)


# ----------------------------------------------------------------------------------
# tokenizer (trained once, committed under tests/golden so token ids are stable)
# ----------------------------------------------------------------------------------
COMMON_WORDS = """the quick brown fox jumped over sleeping dog a an and of to in is it you that he was for on are with as I his
they be at one have this from or had by hot but some what there we can out other were all your when up use word how said each she
which do their time if will way about many then them would write like so these her long make thing see him two has look more day
could go come did my sound no most number who water than call first people may down side been now find any new work part take get
place made live where after back little only round man year came show every good me give our under name very through just form
much great think say help low line before turn cause same mean differ move right boy old too does tell sentence set three want air
well also play small end put home read hand port large spell add even land here must big high such follow act why ask men change
went light kind off need house picture try us again animal point mother world near build self earth father head stand own page
should country found answer school grow study still learn plant cover food sun four thought let keep eye never last door between
city tree cross since hard start might story saw far sea draw left late run while press close night real life few stop open seem
together next white children begin got walk example ease paper often always music those both mark book letter until mile river car
feet care second group carry took rain eat room friend began idea fish mountain north once base hear horse cut sure watch color
face wood main enough plain girl usual young ready above ever red list though feel talk bird soon body family direct pose leave
song measure state product black short numeral class wind question happen complete ship area half rock order fire south problem
piece told knew pass farm top whole king size heard best hour better true during hundred am remember step early hold west ground
interest reach fast five sing listen six table travel less morning ten simple several vowel toward war lay against pattern slow
center love person money serve appear road map science rule govern pull cold notice voice fall power town fine certain fly unit
lead cry dark machine note wait plan figure star box noun field rest correct able pound done beauty drive stood contain front teach
week final gave green oh quick develop sleep warm free minute strong special mind behind clear tail produce fact street inch lot
nothing course stay wheel full force blue object decide surface deep moon island foot yet busy test record boat common gold possible
plane age dry wonder laugh thousand ago ran check game shape yes hot miss brought heat snow bed bring sit perhaps fill east weight
language among speech audio frame model voice stream text token latent decoder transformer kernel memory tensor graph""".split()


def _corpus(seed: int = 7, n_sent: int = 30000) -> list[str]:
    rng = np.random.default_rng(seed)
    onsets = ["", "b", "c", "d", "f", "g", "h", "j", "k", "l", "m", "n", "p", "r", "s", "t", "v", "w", "st", "tr", "ch", "sh", "th", "pl", "br", "gr", "cl"]
    nuclei = ["a", "e", "i", "o", "u", "ai", "ea", "ou", "io", "ee", "oo"]
    codas = ["", "n", "r", "s", "t", "l", "m", "d", "ng", "ck", "st", "nt", "rd"]
    pseudo = []
    for _ in range(4000):
        k = int(rng.integers(1, 4))
        w = "".join(onsets[rng.integers(len(onsets))] + nuclei[rng.integers(len(nuclei))] + codas[rng.integers(len(codas))] for _ in range(k))
        pseudo.append(w)
    vocab = COMMON_WORDS * 6 + pseudo
    puncts = [".", ".", ".", "!", "?", "...", ","]
    out = []
    for _ in range(n_sent):
        n = int(rng.integers(3, 16))
        ws = [vocab[rng.integers(len(vocab))] for _ in range(n)]
        ws[0] = ws[0].capitalize()
        s = ""
        for i, w in enumerate(ws):
            s += w
            if i + 1 < n:
                s += ", " if rng.random() < 0.06 else " "
        s += puncts[rng.integers(len(puncts))]
        if rng.random() < 0.05:
            s = s + " " + str(int(rng.integers(0, 3000)))
        out.append(s)
    out.append("The quick brown fox jumped over the sleeping dog.")
    out.append(".!...?")
    return out


def train_tokenizer(out_model: str) -> None:
    """Unigram, vocab 4000 (reference config.h:69 n_bins=4000), byte fallback, default nmt_nfkc normaliser."""
    import sentencepiece as spm
    import tempfile

    with tempfile.TemporaryDirectory() as td:
        corpus = os.path.join(td, "corpus.txt")
        with open(corpus, "w") as f:
            f.write("\n".join(_corpus()) + "\n")
        prefix = os.path.join(td, "tok")
        spm.SentencePieceTrainer.train(
            input=corpus, model_prefix=prefix, vocab_size=4000, model_type="unigram",
            byte_fallback=True, character_coverage=1.0, num_threads=1,
            input_sentence_size=0, shuffle_input_sentence=False,
            user_defined_symbols=["..."], minloglevel=2,
        )
        shutil.copyfile(prefix + ".model", out_model)


# ----------------------------------------------------------------------------------
def make_model_dir(out_dir: str, seed: int = 1234, dtype: str = "BF16", eos_mode: str = "never",
                   t_voice: int = 125, voices=None, force: bool = False, encoder: bool = False) -> str:
    """Creates (or reuses) the model directory; returns its path WITH trailing '/' (the reference concatenates).
    encoder=True adds the voice-cloning encoder tensors (every other tensor stays bitwise the same)."""
    out_dir = os.path.abspath(out_dir)
    stamp = os.path.join(out_dir, "STAMP.json")
    want = {"seed": seed, "dtype": dtype, "eos_mode": eos_mode, "t_voice": t_voice, "version": 4}
    if encoder:
        want["encoder"] = 1
    if not force and os.path.exists(stamp):
        try:
            if json.load(open(stamp)) == want:
                return out_dir + "/"
        except Exception:
            pass
    os.makedirs(os.path.join(out_dir, "embeddings"), exist_ok=True)
    weights = synth_weights(seed, eos_mode)
    if encoder:
        weights.update(synth_encoder_weights(seed))
    write_safetensors(os.path.join(out_dir, "tts_b6369a24.safetensors"), weights, dtype)
    for v in (voices or VOICES):
        # Voice prompts are always written F32: with a BF16 prompt tensor the reference's residual adds
        # (ggml_add keeps src0's type) would silently run the whole voice prefill in a bf16 residual stream
        # (DESIGN.md "quirks"); the real files' dtype is unknowable offline, so we pin the benign case.
        write_safetensors(os.path.join(out_dir, "embeddings", v + ".safetensors"),
                          {"audio_prompt": synth_voice(v, seed, t_voice)}, "F32")
    if not os.path.exists(GOLDEN_TOKENIZER):
        train_tokenizer(GOLDEN_TOKENIZER)
    shutil.copyfile(GOLDEN_TOKENIZER, os.path.join(out_dir, "tokenizer.model"))
    json.dump(want, open(stamp, "w"))
    return out_dir + "/"


def default_model_dir(eos_mode: str = "never", dtype: str = "BF16", t_voice: int = 125, seed: int = 1234, voices=None, encoder: bool = False) -> str:
    # a cache outside the tree (which may be read-only), one per user: another user's directory on a shared machine is not writable
    root = os.environ.get("PTTS_B200_ASSETS") or os.path.join(tempfile.gettempdir(), f"ptts_b200_assets_{os.getuid()}")
    name = f"model_s{seed}_{dtype.lower()}_{eos_mode + ('7' if eos_mode == 'late' else '')}_v{t_voice}" + ("" if voices is None else "_" + "-".join(voices))
    name += "_enc" if encoder else ""
    return make_model_dir(os.path.join(root, name), seed=seed, dtype=dtype, eos_mode=eos_mode, t_voice=t_voice, voices=voices, encoder=encoder)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--dtype", default="BF16", choices=["BF16", "F32"])
    ap.add_argument("--eos", default="never", choices=["never", "mid", "late"])
    ap.add_argument("--t-voice", type=int, default=125)
    ap.add_argument("--train-tokenizer", action="store_true")
    a = ap.parse_args()
    if a.train_tokenizer:
        train_tokenizer(GOLDEN_TOKENIZER)
        print(GOLDEN_TOKENIZER)
        sys.exit(0)
    if a.out:
        print(make_model_dir(a.out, a.seed, a.dtype, a.eos, a.t_voice, force=True))
    else:
        print(default_model_dir(a.eos, a.dtype, a.t_voice, a.seed))
