"""GPU: the FlowLM attention dispatch in isolation (b200_debug_attention) against a float64 softmax reference, at the edges where the
decomposition of the key space can go wrong: streaming splits and their 8-row stages (including the seam between a shared prefix and a
slot's own rows), shared-prefix tiles of 64 rows with prefix splits (some of them empty when voices have prefixes of different lengths),
the three ways partials are merged, and prefill tile items cut by 64-row runs and by prefill chunks.

Keys and values are written into the cache with b200_debug_write_kv and read back with b200_read_kv, so the reference sees exactly the
bf16 (or f32) values the kernels read; q is passed as f32. Scale 1/8; key k is visible to a row at position pos with prefix length P iff
k < P (from the prefix slot) or P <= k <= pos (from the row's own slot). The row's own rows below P hold poison values that a kernel
reading the wrong slot would pick up.

Two kinds of input, both seeded:
  * random: scores with a standard deviation of ~2.5, so that the softmax is neither uniform nor one-hot (precision);
  * retrieval: every key has norm 8 in every head and q of (row, head) points at one key, or at two keys with equal scores. The output is
    then ~v_target (or the mean of the two), and a key that is dropped, counted twice or taken from the wrong place moves it by O(|v|).
    The targets are the positions where the decomposition has edges (0, P - 1, P, the row's position, split edges, multiples of 8 and
    64 and their neighbours, counted from 0 and from P); a row aims 28 of them per call (4 heads at one key, 12 at two), and a sweep of
    calls aims at every one of them in every row.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

D, H, DH = 1024, 16, 64
KV_CAP = 1600
POISON_V = 50.0

# Tolerances: |out - ref| <= ulp_bf16(ref) + A[path], A in units of the value scale (values ~N(0, 1), |ref| <= ~4).
#  * The output is rounded to bf16 once: half an ulp; the rest of the budget covers an f32 result that sits next to a rounding boundary.
#  * f32-FMA paths (streaming kernel, either cache type): f32 scores and ex2.approx (2^-22 relative) move the pre-rounding value by ~1e-6
#    of |v|; precision 2 (q and probabilities as hi + lo bf16 pairs, ~16 mantissa bits): by ~2^-17 |v| ~ 1e-5.
#  * precision 1 (bf16 probabilities in P V, the sum l in f32): each weight carries up to 2^-9 relative error in the numerator only,
#    <= 2^-9 * max|v| ~ 8e-3 in the worst case; independent per key, so the measured error is well below that.
#  * precision 0 (q also bf16): each score moves by up to 2^-9 * sum_i |q_i k_i| / 8, ~0.06 for a retrieval score of ~25-30, i.e. a few
#    percent of a weight: up to ~0.05 * |v_a - v_b| for a two-target head.
# Measured on a B200 (1000 W power limit; worst over every case of the path, printed by this module with -s), each bound ~4x that:
#   f32 1.3e-6, prec2 8.8e-6, prec1 2.3e-3, prec0 3.5e-2.
TOL = {"f32": 5e-6, "prec2": 3.5e-5, "prec1": 9e-3, "prec0": 1.4e-1}
MEASURED = {}


def _bf16_ulp(x):
    a = np.maximum(np.abs(x), 2.0 ** -126)
    return 2.0 ** (np.floor(np.log2(a)) - 7)


def _check(tag, path, out, ref, rows):
    """Compares the rows `rows` of out with ref; records the absolute term the comparison needed."""
    o, r = out[rows].astype(np.float64), ref[rows]
    assert np.isfinite(o).all(), (tag, "NaN/inf in the output of a live row")
    need = float(np.max(np.abs(o - r) - _bf16_ulp(r)))
    MEASURED[path] = max(MEASURED.get(path, -1.0), need)
    if " retrieval " not in f" {tag} " or "retrieval 0" in tag:                # one line per case: the first retrieval pass and random
        print(f"  [{path}] {tag}: max |err| {np.abs(o - r).max():.3e}, absolute term needed beyond one bf16 ulp {need:.3e} (bound {TOL[path]:.1e})")
    assert need <= TOL[path], (tag, path, need)


def _keys(rng, n, scale=1.0):
    k = rng.standard_normal((n, H, DH))
    k *= 8.0 / np.linalg.norm(k, axis=2, keepdims=True)                   # norm 8 per head: equal scores for equal q . k directions
    return (scale * k).reshape(n, D).astype(np.float32)


class Scene:
    """Rows of one attention call and the cache contents they see, in one engine and layer.
    rows: list of (slot, pos, pfx_slot, P), pos < 0 = dead row; prefixes: {pfx_slot: P}; slots below max_slots get their prefix set."""

    def __init__(self, eng, max_slots, layer, rows, prefixes, seed):
        self.eng, self.max_slots, self.layer, self.rows = eng, max_slots, layer, rows
        rng = np.random.default_rng(seed)
        for ps, P in prefixes.items():
            eng.debug_write_kv(ps, layer, 0, 0, _keys(rng, P))
            eng.debug_write_kv(ps, layer, 1, 0, rng.standard_normal((P, D)).astype(np.float32))
        top = {}
        for slot, pos, ps, P in rows:
            if pos >= 0:
                top[slot] = (max(top.get(slot, (-1, 0))[0], pos), P)
        for slot, (pos, P) in top.items():
            if P > 0:   # own rows below P are never read: poison them
                eng.debug_write_kv(slot, layer, 0, 0, _keys(rng, P, 3.0))
                eng.debug_write_kv(slot, layer, 1, 0, np.full((P, D), POISON_V, np.float32))
            eng.debug_write_kv(slot, layer, 0, P, _keys(rng, pos + 1 - P))
            eng.debug_write_kv(slot, layer, 1, P, rng.standard_normal((pos + 1 - P, D)).astype(np.float32))
        self.apply()
        # what the kernels read: physical rows of the prefix slots and of the own slots (rows >= P), read back from the cache
        self.pfx = {(ps, w): eng.read_kv(ps, layer, w, P).astype(np.float64) for ps, P in prefixes.items() for w in (0, 1)}
        self.own = {(slot, w): eng.read_kv(slot, layer, w, pos + 1).astype(np.float64) for slot, (pos, P) in top.items() for w in (0, 1)}

    def row_kv(self, i, n=None):
        """Keys and values row i sees (float64 [keys][16][64]); n: only the first n of them."""
        slot, pos, ps, P = self.rows[i]
        n = pos + 1 if n is None else n
        kv = []
        for w in (0, 1):
            own = self.own[(slot, w)][P:n]
            kv.append(np.concatenate([self.pfx[(ps, w)][:min(P, n)], own]) if P > 0 else own)
        assert not (np.abs(kv[1]) >= POISON_V).any()
        return kv[0].reshape(-1, H, DH), kv[1].reshape(-1, H, DH)

    def apply(self):
        for slot, pos, ps, P in self.rows:
            if slot < self.max_slots:
                self.eng.debug_set_prefix(slot, ps if P > 0 else 0, P)

    def live(self):
        return [i for i, r in enumerate(self.rows) if r[1] >= 0]

    def reference(self, q, drop=None):
        """float64 softmax attention; drop = {(row, head): key} removes one key from that (row, head). Rows of one slot share a pass."""
        out = np.zeros((len(self.rows), D))
        groups = {}
        for i in self.live():
            groups.setdefault(self.rows[i][0], []).append(i)
        for rows in groups.values():
            top = max(rows, key=lambda i: self.rows[i][1])
            K, V = self.row_kv(top)
            pos = np.array([self.rows[i][1] for i in rows])
            s = np.einsum("lhd,rhd->rhl", K, q[rows].reshape(len(rows), H, DH).astype(np.float64)) / 8.0
            s = np.where(np.arange(K.shape[0])[None, None, :] > pos[:, None, None], -np.inf, s)   # causal: key <= the row's position
            if drop:
                for r, i in enumerate(rows):
                    for h in range(H):
                        if (i, h) in drop:
                            s[r, h, drop[(i, h)]] = -np.inf
            p = np.exp(s - s.max(axis=2, keepdims=True))
            p /= p.sum(axis=2, keepdims=True)
            out[rows] = np.einsum("rhl,lhd->rhd", p, V).reshape(len(rows), D)
        return out

    def random_q(self, seed):
        rng = np.random.default_rng(seed)
        return (2.5 * rng.standard_normal((len(self.rows), D))).astype(np.float32)   # score sd = 2.5 with |k| = 8 per head

    PER_PASS = 4 + 2 * (H - 4)                                           # 4 single-target heads, 12 two-target heads

    def retrieval_sweep(self, splits=(), gamma=3.0):
        """Yields (q, {(row, head): single target}) passes that together aim at EVERY boundary key of every row (_targets): pass j takes
        targets [28 j, 28 j + 28) of each row's list, a row whose list is used up takes its first targets again. Asserts the coverage."""
        tl = {i: _targets(self.rows[i][3], self.rows[i][1], splits, rot=i) for i in self.live()}
        passes = max(-(-len(t) // self.PER_PASS) for t in tl.values())
        hit = {i: set() for i in tl}
        for j in range(passes):
            q = np.zeros((len(self.rows), D), np.float32)
            single = {}
            for i, t in tl.items():
                slot, pos, ps, P = self.rows[i]
                pick = [t[(j * self.PER_PASS + u) % len(t)] for u in range(self.PER_PASS)]
                hit[i].update(pick)
                key = lambda k, h: (self.pfx[(ps, 0)][k] if k < P else self.own[(slot, 0)][k]).reshape(H, DH)[h]
                u = 0
                for h in range(H):
                    a = pick[u]; u += 1
                    if h < 4:
                        v = key(a, h); single[(i, h)] = a
                    else:
                        b = pick[u]; u += 1
                        v = key(a, h) + key(b, h) if b != a else key(a, h)
                    q[i, h * DH:(h + 1) * DH] = gamma * v
            yield q, single
        assert all(hit[i] == set(t) for i, t in tl.items())

    def retrieval_q(self, splits=(), gamma=3.0):
        """The first pass of retrieval_sweep."""
        return next(self.retrieval_sweep(splits, gamma))


def _targets(P, pos, splits, rot):
    """Key positions of a row where the key-space decomposition has edges: most specific first, the periodic ones rotated by `rot`."""
    L = pos + 1
    first = [pos, P, P - 1, 0, pos - 1, P + 1, 1]
    for sp in splits:                                                    # streaming split edges, prefix streamed or reduced elsewhere
        for ntot, base in ((L, 0), (L - P, P)):
            chunk = -(-(-(-ntot // sp)) // 8) * 8
            for c in range(1, sp):
                first += [base + c * chunk - 1, base + c * chunk]
    periodic = [k for k in range(L) if k % 8 in (0, 7) or (k - P) % 8 in (0, 7) or k % 64 == 1 or (k - P) % 64 == 1]
    if periodic:
        r = (rot * 29) % len(periodic)
        periodic = periodic[r:] + periodic[:r]
    out = []
    for k in first + periodic:
        if 0 <= k <= pos and k not in out:
            out.append(k)
    return out


def _inputs(sc, splits, seed):
    """Every pass of the retrieval sweep, then one random input."""
    for j, (q, _) in enumerate(sc.retrieval_sweep(splits)):
        yield f"retrieval {j}", q
    yield "random", sc.random_q(seed)


def _run(eng, scene, q, prefill=False, slot0=0, **opts):
    rows_pos = [r[1] for r in scene.rows]
    rows_slot = [r[0] for r in scene.rows] if prefill else None
    out, tiles = eng.debug_attention(scene.layer, q, rows_pos, slot0=slot0, rows_slot=rows_slot, prefill=prefill, **opts)
    return out, tiles


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx_bf16(P, model_dir):
    c = P.Context(model_dir, max_slots=160, max_voices=8, kv_capacity=KV_CAP)
    yield c
    c.close()


def _decode_stream_rows(S, slot0, rng):
    """Streaming-only decode rows: private caches from 1 to 1501 keys, shared prefixes with P % 8 in {0, 1, 7} (an 8-row stage spans
    the seam between the prefix and the own rows), small prefixes, suffixes of a single key, dead rows."""
    rows, prefixes = [], {S + 4: 1345, S + 5: 1344, S + 6: 1343, S + 7: 125, S + 3: 1}
    slot = slot0
    for pos in (0, 3, 7, 8, 9, 63, 64, 65, 200, 777, 1500):
        rows.append((slot, pos, 0, 0)); slot += 1
    for ps, P in prefixes.items():
        for suf in (0, 1, 7, 8, int(rng.integers(9, 140))):
            rows.append((slot, P + suf, ps, P)); slot += 1
    rows.insert(5, (slot, -1, 0, 0)); slot += 1
    rows.insert(20, (slot, -1, S + 4, 1345)); slot += 1
    # slots must be slot0 + r
    return [(slot0 + i, pos, ps, P) for i, (_, pos, ps, P) in enumerate(rows)], prefixes


@pytest.fixture(scope="module")
def stream_scene(ctx_bf16):
    S = 160
    rows, prefixes = _decode_stream_rows(S, 112, np.random.default_rng(5))
    return Scene(ctx_bf16.engine, 160, 0, rows, prefixes, seed=11)


@pytest.mark.parametrize("splits", [1, 2, 3, 16])
def test_decode_streaming_bf16(ctx_bf16, stream_scene, splits):
    eng, sc = ctx_bf16.engine, stream_scene
    sc.apply()
    live = sc.live()
    slot0 = sc.rows[0][0]
    for kind, q in _inputs(sc, (splits,), splits):
        out, tiles = _run(eng, sc, q, slot0=slot0, stream_splits=splits, tile_min_rows=1 << 20)
        assert tiles == 0
        _check(f"decode stream bf16 splits={splits} {kind}", "f32", out, sc.reference(q), live)
        dead = [i for i, r in enumerate(sc.rows) if r[1] < 0]
        assert np.isnan(out[dead]).all()                                  # nothing is written for a dead row
        out2, _ = _run(eng, sc, q, slot0=slot0, stream_splits=splits, tile_min_rows=1 << 20)
        assert np.array_equal(out, out2, equal_nan=True)                  # deterministic


def test_decode_streaming_row_independent_of_batch(ctx_bf16, stream_scene):
    """With a fixed split count a row's keys are cut the same way whatever else is in the batch: bitwise the same output alone."""
    eng, sc = ctx_bf16.engine, stream_scene
    sc.apply()
    q = sc.random_q(7)
    out, _ = _run(eng, sc, q, slot0=sc.rows[0][0], stream_splits=3, tile_min_rows=1 << 20)
    for i in sc.live()[::3]:
        alone, _ = eng.debug_attention(sc.layer, q[i:i + 1], [sc.rows[i][1]], slot0=sc.rows[i][0], stream_splits=3, tile_min_rows=1 << 20)
        assert np.array_equal(alone[0], out[i]), i


def test_retrieval_is_discriminative(ctx_bf16, stream_scene):
    """The margin of the retrieval inputs: without its target key, a single-target head's reference moves far beyond the tolerance."""
    eng, sc = ctx_bf16.engine, stream_scene
    sc.apply()
    q, single = sc.retrieval_q(splits=(3,))
    single = {(i, h): k for (i, h), k in single.items() if sc.rows[i][1] > 0}   # a row with one key keeps it
    out, _ = _run(eng, sc, q, slot0=sc.rows[0][0], stream_splits=3, tile_min_rows=1 << 20)
    ref = sc.reference(q)
    gone = sc.reference(q, drop=single)
    worst = np.inf
    for (i, h), k in single.items():
        sl = slice(h * DH, (h + 1) * DH)
        tol = float(np.max(_bf16_ulp(ref[i, sl]) + TOL["f32"]))
        worst = min(worst, float(np.max(np.abs(gone[i, sl] - out[i, sl]))) / tol)
    print(f"  retrieval margin: a dropped target moves a head by >= {worst:.0f}x its tolerance")
    assert worst > 20.0


# ---- shared-prefix tiles ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tile_scene(ctx_bf16):
    """One decode batch: voices with prefixes of 1345, 125, 64 and 1 rows (the split count follows the longest, so the short prefixes
    have empty splits), 70 rows of the first voice (a full 64-row tile and a ragged one), voices interleaved by slot, private rows, dead
    rows, rows whose own suffix is a single key."""
    S = 160
    rng = np.random.default_rng(3)
    prefixes = {S + 4: 1345, S + 5: 125, S + 6: 64, S + 7: 1}
    kinds = [S + 4] * 70 + [S + 5] * 12 + [S + 6] * 9 + [S + 7] * 7 + [0] * 6 + [-1] * 6
    rng.shuffle(kinds)
    rows, first = [], set()
    for r, ps in enumerate(kinds):
        if ps == -1:
            rows.append((r, -1, S + 4, 1345))                                  # dead row of a voice: inside the voice's tile, never merged
        elif ps == 0:
            rows.append((r, int(rng.integers(0, 300)), 0, 0))
        else:
            P = prefixes[ps]
            suf = 0 if ps not in first else int(rng.integers(0, 150))
            first.add(ps)
            rows.append((r, P + suf, ps, P))
    return Scene(ctx_bf16.engine, 160, 2, rows, prefixes, seed=13)


@pytest.mark.parametrize("prec", [0, 1, 2])
def test_decode_prefix_tiles(ctx_bf16, tile_scene, prec):
    eng, sc = ctx_bf16.engine, tile_scene
    sc.apply()
    live = sc.live()
    dead = [i for i, r in enumerate(sc.rows) if r[1] < 0]
    path = {0: "prec0", 1: "prec1", 2: "prec2"}[prec]
    for kind, q in _inputs(sc, (3,), 100 + prec):
        ref = sc.reference(q)
        outs = {}
        for name, opts in (("merge kernel", dict(fork_tiles=1, counted_merge=0)), ("counted merge", dict(fork_tiles=1, counted_merge=1)),
                           ("in-kernel merge", dict(fork_tiles=0, counted_merge=0))):
            out, tiles = _run(eng, sc, q, tile_prec=prec, stream_splits=3, tile_min_rows=4, **opts)
            assert tiles == 1
            _check(f"decode prefix tiles, {name}, {kind}", path, out, ref, live)
            assert np.isnan(out[dead]).all()
            outs[name] = out
        # the counted merge combines the same partials in the same order with the same arithmetic as attn_merge_kernel
        assert np.array_equal(outs["merge kernel"], outs["counted merge"], equal_nan=True)
        again, _ = _run(eng, sc, q, tile_prec=prec, stream_splits=3, tile_min_rows=4, fork_tiles=1, counted_merge=0)
        assert np.array_equal(outs["merge kernel"], again, equal_nan=True)


def test_debug_attention_refuses_oversized_work_list(ctx_bf16, tile_scene):
    """More distinct prefixes than the prefix-tile work list holds (it is sized for max_voices of them): an error, not an abort."""
    eng = ctx_bf16.engine
    for r in range(110):
        eng.debug_set_prefix(r, 160 + 4, 1 + r)                           # 110 prefixes of different lengths -> 110 one-split items
    with pytest.raises(RuntimeError, match="-5"):
        eng.debug_attention(0, np.zeros((110, D), np.float32), [200] * 110, slot0=0)
    tile_scene.apply()


def test_decode_prefix_tiles_engine_defaults(ctx_bf16, tile_scene):
    """The options a step runs with (automatic split count, default precision and merge)."""
    eng, sc = ctx_bf16.engine, tile_scene
    sc.apply()
    q = sc.retrieval_q()[0]
    out, tiles = _run(eng, sc, q)
    assert tiles == 1
    _check("decode prefix tiles, engine defaults, retrieval", "prec1", out, sc.reference(q), sc.live())


# ---- prefill ----------------------------------------------------------------------------------------------------------------------
def _prefill_rows(S, base):
    """Slot-major rows: a voice prefill (P = 0 from position 0), sentences after shared prefixes of 1345 and 125 rows, one after a
    private copy of a 125-row prefix, and a one-token sentence after a 64-row prefix. Sentences longer than 64 tokens."""
    prefixes = {S + 4: 1345, S + 5: 125, S + 6: 64}
    rows = []
    rows += [(base + 0, p, S + 4, 1345) for p in range(1345, 1345 + 100)]
    rows += [(base + 1, p, S + 5, 125) for p in range(125, 125 + 130)]
    rows += [(base + 2, p, 0, 0) for p in range(125, 125 + 70)]
    rows += [(base + 3, 64, S + 6, 64)]
    rows += [(S + 3, p, 0, 0) for p in range(0, 140)]
    return rows, prefixes


def _prefill_case(eng, S, chunk, layer, base, seed, precs, path_of):
    rows, prefixes = _prefill_rows(S, base)
    sc = Scene(eng, S, layer, rows, prefixes, seed=seed)
    for prec in precs:
        for kind, q in _inputs(sc, (), seed + prec):
            out, items = _run(eng, sc, q, prefill=True, prefill_prec=prec)
            _check(f"prefill chunk={chunk} prec={prec} {kind} ({items} tile items)", path_of(prec), out, sc.reference(q), sc.live())
            again, _ = _run(eng, sc, q, prefill=True, prefill_prec=prec)
            assert np.array_equal(out, again)


@pytest.mark.parametrize("chunk", [64, 100, 4096])
def test_prefill_tiles(P, model_dir, ctx_bf16, chunk):
    """Tile items of <= 64 positions per slot, built per chunk: chunks of 64 and 100 rows cut sentences and 64-row runs."""
    own = chunk != 4096
    c = P.Context(model_dir, max_slots=8, max_voices=8, kv_capacity=KV_CAP, max_prefill_rows=chunk) if own else ctx_bf16
    S, base = (8, 0) if own else (160, 152)
    try:
        _prefill_case(c.engine, S, chunk, 5, base, 40 + chunk, (2, 1, 0) if not own else (2,), lambda p: f"prec{p}")
    finally:
        if own:
            c.close()


# ---- f32 cache: streaming kernel only (decode and prefill) ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx_f32(P, model_dir):
    c = P.Context(model_dir, max_slots=48, max_voices=8, kv_capacity=KV_CAP, kv_f32=1, max_prefill_rows=100)
    yield c
    c.close()


@pytest.mark.parametrize("splits", [1, 2, 3, 16])
def test_decode_streaming_f32(ctx_f32, splits):
    eng = ctx_f32.engine
    rows, prefixes = _decode_stream_rows(48, 0, np.random.default_rng(6))
    sc = Scene(eng, 48, 1, rows, prefixes, seed=17 + splits)
    for kind, q in _inputs(sc, (splits,), splits):
        out, tiles = _run(eng, sc, q, stream_splits=splits)
        assert tiles == 0
        _check(f"decode stream f32 splits={splits} {kind}", "f32", out, sc.reference(q), sc.live())


def test_prefill_streaming_f32(ctx_f32):
    """f32 cache: prefill rows go through the streaming kernel one row per CTA, in chunks of 100 rows."""
    _prefill_case(ctx_f32.engine, 48, 100, 4, 0, 77, (2,), lambda p: "f32")


def test_zz_report_measured():
    """Summary of the worst absolute terms measured per path (printed with -s)."""
    print("\n[attention] absolute term needed beyond one bf16 ulp, worst per path: " +
          ", ".join(f"{k} {v:.2e} (bound {TOL[k]:.0e})" for k, v in sorted(MEASURED.items())))
