"""GPU: per-sentence sampling controls (DESIGN.md 4.7): LSD decode steps, truncated noise and the EOS threshold.

- A sentence begun with explicit default controls runs exactly today's step: same graphs, same launch count, bitwise the same PCM,
  latents and EOS logits (bench-shaped batch with overlap 0 / 1, the batch-1 persistent path, Batch.run()).
- Rows with default controls in a batch whose other rows use N = 4 and the clamp are bitwise equal to an all-default run.
- The N-step head agrees with a float64 restatement (out_norm -> cond -> N-step LSD, the engine's bf16 rounding points) at R = 1, 2, 3,
  64 and 256 (fused cluster kernel from 3 rows on, unfused chain below and with taps on).
- The truncated draws stay inside [-a, a], match the truncated normal's moments and CDF, and depend on (seed, stream id, step) only.
- The stop frame follows the threshold: first frame with logit > tau, plus frames_after_eos; at tau = -4 the golden frame counts.
"""
import json
import os

import numpy as np
import pytest

from conftest import REPO

pytestmark = pytest.mark.gpu
GOLD = os.path.join(REPO, "tests", "golden")
DEFAULT = (1, 0.0, -4.0)
# latent vs the float64 restatement (DESIGN.md §2): N = 1 keeps the existing latent tolerance, N > 1 is ~4x the worst value measured on a B200
HEAD_MAXABS, HEAD_REL_N1, HEAD_REL = 4e-2, 1.5e-2, 8e-3


@pytest.fixture(scope="module")
def bench_dir():
    from make_assets import default_model_dir
    return default_model_dir(eos_mode="never", t_voice=1345, voices=["cosette"])


def _run_steps(P, eng, B, frames):
    pcm, lat, eos, launches = [], [], [], []
    for _ in range(frames):
        l0 = eng.launch_count()
        p, prod, la, eo = eng.step(0, B, None)
        launches.append(eng.launch_count() - l0)
        pcm.append(p); lat.append(la); eos.append(eo)
    return np.stack(pcm), np.stack(lat), np.stack(eos), launches


def _begin(eng, B, voice, toks, mg, sampling):
    eng.begin_sentences(list(range(B)), [voice] * B, toks, mg, [1 << 20] * B, [0.7] * B, rng_streams=list(range(1, B + 1)), sampling=sampling)


@pytest.mark.parametrize("overlap", [0, 1])
def test_default_controls_run_todays_step(overlap, P, bench_dir):
    import bench
    B, frames = 256, 20
    ctx = P.Context(bench_dir, max_slots=B, max_voices=1, kv_capacity=2048, overlap=overlap)
    eng = ctx.engine
    voice = ctx.stream("cosette", temp=0.7).voice
    toks = [ctx.tokenize(bench.synth_paragraph(i)) for i in range(B)]
    runs = []
    for sampling in (None, [DEFAULT] * B, None, [DEFAULT] * B):          # second pair: both replay captured graphs
        eng.set_seed(11)
        _begin(eng, B, voice, toks, [200] * B, sampling)
        runs.append(_run_steps(P, eng, B, frames))
    for a, b in ((runs[0], runs[1]), (runs[2], runs[3]), (runs[0], runs[2])):
        for x, y in zip(a[:3], b[:3]):
            assert np.array_equal(x, y)
        assert a[3] == b[3]
    assert np.isfinite(runs[0][0]).all()


def test_default_controls_batch1_and_batch_run(P, model_dir):
    ctx = P.Context(model_dir, max_slots=1, kv_capacity=512)
    eng = ctx.engine
    voice = ctx.stream("cosette", temp=0.7).voice
    toks = [ctx.tokenize("The quick brown fox jumped over the sleeping dog.")]
    runs = []
    for sampling in (None, [DEFAULT], None, [DEFAULT]):
        eng.set_seed(3)
        _begin(eng, 1, voice, toks, [60], sampling)
        runs.append(_run_steps(P, eng, 1, 20))
    for a in runs[1:]:
        for x, y in zip(a[:3], runs[0][:3]):
            assert np.array_equal(x, y)
        assert a[3] == runs[0][3]
    ctx.close()

    texts = ["Hello world.", "One two three four five six seven eight nine ten eleven twelve.", "Short one.", "How are you today my friend?"]
    reads = []
    for kw in ({}, dict(lsd_steps=1, noise_clamp=0.0, eos_threshold=-4.0)):
        c = P.Context(model_dir, max_slots=4, max_voices=1, kv_capacity=512)
        P.set_seed(9)
        b = P.Batch(c, 4)
        utts = [b.add("cosette", t, 0.7, **kw) for t in texts]
        b.run()
        reads.append([b.read(u) for u in utts])
        del b
        c.close()
    for x, y in zip(*reads):
        assert np.array_equal(x, y)


def test_mixed_batch_does_not_leak(P, model_dir):
    B = 16
    ctx = P.Context(model_dir, max_slots=B, max_voices=1, kv_capacity=512)
    eng = ctx.engine
    voice = ctx.stream("cosette", temp=0.7).voice
    toks = [ctx.tokenize(f"Sentence number {i} is spoken here with a few more words.") for i in range(B)]
    custom = [i % 2 == 1 for i in range(B)]
    out = {}
    for name, sampling in (("default", [DEFAULT] * B), ("mixed", [(4, 0.3, -4.0) if c else DEFAULT for c in custom])):
        eng.set_seed(5)
        _begin(eng, B, voice, toks, [100] * B, sampling)
        out[name] = _run_steps(P, eng, B, 12)
    d, m = out["default"], out["mixed"]
    for x, y in zip(d[:3], m[:3]):
        assert np.array_equal(x[:, ~np.array(custom)], y[:, ~np.array(custom)])
    assert np.isfinite(m[0]).all() and not np.array_equal(d[1][:, 1], m[1][:, 1])


# ---- float64 restatement of the head (engine rounding points: bf16 GEMM operands, f32 elsewhere) ----
def _bf(x):
    x = np.asarray(x, np.float32)
    b = x.view(np.uint32).astype(np.uint64)
    r = ((b + 0x7FFF + ((b >> 16) & 1)) >> 16) << 16
    return r.astype(np.uint32).view(np.float32).astype(np.float64)


def _silu(x):
    return x / (1.0 + np.exp(-x))


def _ln(x, w, b, eps):
    m = x.mean(-1, keepdims=True)
    v = ((x - m) ** 2).mean(-1, keepdims=True)
    y = (x - m) / np.sqrt(v + eps)
    return y * (w if w is not None else 1.0) + (b if b is not None else 0.0)


class HeadRef:
    def __init__(self, model_dir):
        from make_assets import read_safetensors
        W = read_safetensors(os.path.join(model_dir, "tts_b6369a24.safetensors"))
        self.W = {k: np.asarray(v, np.float64) for k, v in W.items()}
        self.f = "flow_lm.flow_net."

    def lin(self, name, x):
        y = _bf(x) @ _bf(self.W[name + ".weight"]).T
        b = self.W.get(name + ".bias")
        return y + b if b is not None else y

    def tcomb(self, s, t):
        out = 0.0
        for idx, tv in ((0, s), (1, t)):
            p = self.f + f"time_embed.{idx}."
            a = (self.W[p + "freqs"].astype(np.float32) * np.float32(tv)).astype(np.float64)
            e = _bf(np.concatenate([np.cos(a), np.sin(a)]))
            h1 = _bf(_silu(e @ _bf(self.W[p + "mlp.0.weight"]).T + self.W.get(p + "mlp.0.bias", 0.0)))
            u = h1 @ _bf(self.W[p + "mlp.2.weight"]).T + self.W.get(p + "mlp.2.bias", 0.0)
            out = out + self.W[p + "mlp.3.alpha"] * u / np.sqrt(u.var(ddof=1) + 1e-5)
        return out / 2

    def head(self, h, noise, N):
        W, f = self.W, self.f
        c = _ln(h, W["flow_lm.out_norm.weight"], W.get("flow_lm.out_norm.bias"), 1e-5)
        cond = self.lin(f + "cond_embed", c)
        x = noise.astype(np.float64)
        for i in range(N):
            sy = _silu(cond + self.tcomb(np.float32(i) / np.float32(N), np.float32(i + 1) / np.float32(N)))
            xr = self.lin(f + "input_proj", x)
            for r in range(6):
                p = f + f"res_blocks.{r}."
                sh, sc, g = np.split(self.lin(p + "adaLN_modulation.1", sy), 3, axis=-1)
                a = _ln(xr, W.get(p + "in_ln.weight"), W.get(p + "in_ln.bias"), 1e-6) * (1 + sc) + sh
                xr = xr + g * self.lin(p + "mlp.2", _silu(self.lin(p + "mlp.0", a)))
            sh, sc = np.split(self.lin(f + "final_layer.adaLN_modulation.1", sy), 2, axis=-1)
            a = _ln(xr, W.get(f + "final_layer.norm_final.weight"), W.get(f + "final_layer.norm_final.bias"), 1e-6) * (1 + sc) + sh
            x = x + self.lin(f + "final_layer.linear", a) / N
        return x


@pytest.fixture(scope="module")
def head_ref(model_dir):
    return HeadRef(model_dir)


@pytest.mark.parametrize("R", [1, 2, 3, 64, 256])
def test_multistep_head_matches_restatement(R, P, model_dir, head_ref):
    ctx = P.Context(model_dir, max_slots=R, max_voices=1, kv_capacity=256)
    eng = ctx.engine
    voice = ctx.stream("cosette", temp=0.7).voice
    toks = [ctx.tokenize(f"Row {i} says a short sentence.") for i in range(R)]
    rng = np.random.default_rng(R)
    for N in (1, 2, 3, 8):
        noise = (rng.standard_normal((R, 32)) * np.sqrt(0.7)).astype(np.float32)
        lat = {}
        for taps in (1, 0):                                               # taps on: unfused chain at every R; off: fused from 3 rows
            eng.debug_taps(taps == 1)
            _begin(eng, R, voice, toks, [50] * R, [(N, 0.0, -4.0)] * R)
            _, prod, lat[taps], _ = eng.step(0, R, noise)
            assert prod.all()
            if taps:
                h = np.stack([eng.debug_tap("flow.layer5", r) for r in range(R)])
        eng.debug_taps(False)
        ref = head_ref.head(h.astype(np.float64), noise, N)
        for taps, got in lat.items():
            err = float(np.abs(got - ref).max()); rel = float(np.linalg.norm(got - ref) / np.linalg.norm(ref))
            assert err < HEAD_MAXABS and rel < (HEAD_REL_N1 if N == 1 else HEAD_REL), (R, N, taps, err, rel)


def _drawn(eng, R):
    eng.sync()
    return eng.debug_read("noise_drawn", 0, R * 32).reshape(R, 32)


@pytest.mark.parametrize("k", [0.3, 1.0, 2.0])
def test_truncated_noise_distribution(k, P, model_dir):
    from scipy import stats
    R, temp = 256, 0.7
    sigma = float(np.sqrt(np.float32(temp)))
    a = float(np.float32(k * sigma))
    ctx = P.Context(model_dir, max_slots=R, max_voices=1, kv_capacity=1024)
    eng = ctx.engine
    voice = ctx.stream("cosette", temp=temp).voice
    toks = [ctx.tokenize("A sentence.")] * R
    eng.set_seed(21)
    # slots 0 and 1 share the RNG stream id: the same draws in different slots
    rs = [1000, 1000] + list(range(2, R))
    eng.begin_sentences(list(range(R)), [voice] * R, toks, [400] * R, [1 << 20] * R, [temp] * R, rng_streams=rs, sampling=[(1, a, -4.0)] * R)
    draws = []
    for _ in range(125):                                                  # 125 x 256 x 32 = 1.02e6 draws
        eng.step_enqueue(0, R)
        z = _drawn(eng, R)
        assert np.array_equal(z[0], z[1])
        draws.append(z[2:].ravel())
    z = np.concatenate(draws).astype(np.float64)
    assert z.size >= 10 ** 6
    assert np.abs(z).max() <= a
    lo, hi = -a / sigma, a / sigma
    tn = stats.truncnorm(lo, hi, scale=sigma)
    m_err = abs(z.mean() - tn.mean()) / np.sqrt(tn.var() / z.size)
    v_err = abs(z.var() - tn.var()) / tn.var()
    ks = stats.kstest(z, tn.cdf)
    assert m_err < 5.0 and v_err < 6e-3 and ks.pvalue > 1e-4, (m_err, v_err, ks.pvalue)


def test_eos_threshold_moves_the_stop_frame(P, model_dir_eos, oracle_mod):
    counts = json.load(open(os.path.join(GOLD, "frame_counts_eos_mid.json")))
    c = P.Context(model_dir_eos, max_slots=1, kv_capacity=1024)
    st = c.stream("cosette", temp=0.7)
    eng = c.engine

    def run(text, info, tau):
        toks = c.tokenize(text)
        mg, fae = oracle_mod.max_gen_len_for(text), oracle_mod.frames_after_eos_guess(text)
        eng.begin_sentences([st.slot], [st.voice], [toks], [mg], [fae], [0.7], sampling=[(1, 0.0, tau)])
        rng = np.random.default_rng(info["seed"])
        logits = []
        while True:
            noise = (rng.standard_normal(32) * np.sqrt(0.7)).astype(np.float32)
            _, prod, _, eo = eng.step(st.slot, 1, noise[None])
            if not prod[0]:
                return len(logits), logits, mg, fae
            logits.append(float(eo[0]))
            assert len(logits) <= mg

    checked = 0
    for text, info in counts.items():
        n, logits, mg, fae = run(text, info, -4.0)
        assert n == info["frames"], text
        lg = np.array(logits, np.float32)
        vals = np.unique(lg)
        taus = [float(np.float32((x + y) / 2) - np.float32(4)) for x, y in zip(vals[:-1], vals[1:])]
        for tau in taus[:: max(1, len(taus) // 3)][:3]:
            above = np.nonzero(lg > np.float32(tau) + np.float32(4))[0]
            if not len(above):
                continue
            n_tau, _, _, _ = run(text, info, tau)
            assert n_tau == min(int(above[0]) + fae, mg), (text, tau, n_tau, int(above[0]))
            checked += 1
    assert checked >= 3
