"""Float64 numpy restatement of the resampler in front of the voice-cloning encoder (DESIGN.md §4.6): torchaudio.functional.resample(x,
sr, 24000) with its defaults (sinc_interp_hann, lowpass_filter_width 6, rolloff 0.99), computed over each phase's band of nonzero taps
instead of torchaudio's dense [m][2w + o] kernel, so that any integer rate fits in memory."""
import math

import numpy as np

SR = 24000
L = 6                      # lowpass_filter_width
ROLLOFF = 0.99


def plan(sr: int) -> dict:
    """o / m: the reduced rates; w: torchaudio's kernel width; X: |(k - w) m - i o| <= X is the band of phase i (exact integers); W: the
    widest band; lo[i]: the first tap of phase i, as k - w."""
    g = math.gcd(sr, SR)
    o, m = sr // g, SR // g
    base = min(o, m) * ROLLOFF
    w = math.ceil(L * o / base)
    X = 600 * max(o, m) // 99
    i = np.arange(m, dtype=np.int64)
    lo = -((X - i * o) // m)             # ceil((i o - X) / m)
    hi = (i * o + X) // m
    return {"sr": sr, "o": o, "m": m, "base": base, "w": w, "X": X, "W": int((hi - lo + 1).max()), "lo": lo, "hi": hi}


def out_len(n: int, sr: int) -> int:
    """n24 = ceil(24000 n / sr)."""
    return -(-n * SR // sr)


def kernel(p: dict, i, d) -> np.ndarray:
    """K[i][w + d] in float64, in torchaudio's operation order (i, d broadcast)."""
    t = (-np.asarray(i, np.float64)) / p["m"] + np.asarray(d, np.float64) / p["o"]
    t = t * p["base"]
    t = np.clip(t, -L, L)
    window = np.cos(t * math.pi / L / 2) ** 2
    t = t * math.pi
    with np.errstate(invalid="ignore", divide="ignore"):
        k = np.where(t == 0, 1.0, np.sin(t) / np.where(t == 0, 1.0, t))
    return k * (window * (p["base"] / p["o"]))


def band_table(p: dict) -> np.ndarray:
    """coef [m][W] float64: coef[i][b] = K[i][w + lo[i] + b], 0 past the phase's band or outside torchaudio's taps 0 .. 2w + o - 1."""
    i = np.arange(p["m"])[:, None]
    d = p["lo"][:, None] + np.arange(p["W"])[None, :]
    ok = (d <= p["hi"][:, None]) & (d >= -p["w"]) & (d < p["w"] + p["o"])
    return np.where(ok, kernel(p, i, d), 0.0)


def dense_from_band(p: dict, coef: np.ndarray) -> np.ndarray:
    """The band table scattered into torchaudio's dense layout [m][2w + o]."""
    out = np.zeros((p["m"], 2 * p["w"] + p["o"]), coef.dtype)
    for i in range(p["m"]):
        for b in range(p["W"]):
            k = p["w"] + p["lo"][i] + b
            if 0 <= k < out.shape[1]:
                out[i, k] = coef[i, b]
            else:
                assert coef[i, b] == 0
    return out


def resample(x, sr: int, f32_table: bool = False) -> np.ndarray:
    """x (any float dtype) at sr Hz -> float64 [n24] at 24 kHz. f32_table: the coefficients rounded to f32 first, as the device uses them
    (the sum stays float64)."""
    x = np.asarray(x, np.float64).reshape(-1)
    if sr == SR:
        return x.copy()
    p = plan(sr)
    coef = band_table(p)
    if f32_table:
        coef = coef.astype(np.float32).astype(np.float64)
    n, n24 = len(x), out_len(len(x), sr)
    j = np.arange(n24, dtype=np.int64)
    q, i = j // p["m"], j % p["m"]
    s = q * p["o"] + p["lo"][i]          # first input sample of output j
    y = np.zeros(n24)
    for b in range(p["W"]):
        g = s + b
        ok = (g >= 0) & (g < n)
        y += coef[i, b] * np.where(ok, x[np.clip(g, 0, max(n - 1, 0))], 0.0)
    return y


def encoder_input(x, sr: int) -> np.ndarray:
    """What the encoder reads: the 24 kHz signal (f32-rounded coefficients), zero-padded to 1920 T."""
    y = resample(x, sr, f32_table=True)
    T = -(-len(y) // 1920)
    return np.concatenate([y, np.zeros(1920 * T - len(y))])
