"""numpy restatement of `lsd_degrade_audio` (csrc/audio_degrade.cu): the counter-based generator, the synthetic room impulse
response, white noise at an SNR, overdrive clipping, the band limit (`scipy.signal.resample_poly` down and up, with taps built as
`firwin` builds them) and the G.711 mu-law round trip of CPython's `audioop`.  Every stage works on float64 except where the
device's own float32 arithmetic is stated (clip, mu-law), so the tests can compare those bit for bit and the others within a
tolerance.

Stages run in the order reverb, noise, clip, band, mu-law; a variant enables each with one bit."""
from __future__ import annotations

import numpy as np

SR = 16000
REVERB, NOISE, CLIP, BAND, MULAW = 1, 2, 4, 8, 16
STREAM_NOISE, STREAM_RIR = 0, 1
_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _splitmix64(z: np.ndarray) -> np.ndarray:
    z = z.astype(np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def random_bits(seed: int, stream: int, idx: np.ndarray) -> np.ndarray:
    """64 random bits for sample indices `idx` of (seed, stream): splitmix64(splitmix64(seed << 32 | stream) + idx)."""
    key = _splitmix64(np.array([(int(seed) << 32) | int(stream)], dtype=np.uint64))[0]
    with np.errstate(over="ignore"):
        return _splitmix64(np.asarray(idx, dtype=np.uint64) + key)


def uniforms24(seed: int, stream: int, idx: np.ndarray):
    """The two 24-bit integers of every draw: u1 from bits 40..63, u2 from bits 16..39."""
    r = random_bits(seed, stream, idx)
    return (r >> np.uint64(40)).astype(np.int64), ((r >> np.uint64(16)) & np.uint64(0xFFFFFF)).astype(np.int64)


def gaussian(seed: int, stream: int, idx: np.ndarray) -> np.ndarray:
    """Box-Muller in double: sqrt(-2 ln((a + 1) / 2^24)) * cos(2 pi b / 2^24)."""
    a, b = uniforms24(seed, stream, idx)
    u1 = (a + 1).astype(np.float64) * 2.0 ** -24
    u2 = b.astype(np.float64) * 2.0 ** -24
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def rir_length(rt60: float) -> int:
    return int(np.rint(float(np.float32(rt60)) * SR))


def rir(rt60: float, seed: int) -> np.ndarray:
    """h[0] = 1; h[j] = g_j 10^(-3 j / L) for 1 <= j < L, the tail scaled to unit energy (direct-to-reverberant ratio 0 dB)."""
    L = rir_length(rt60)
    j = np.arange(1, L, dtype=np.int64)
    tail = gaussian(seed, STREAM_RIR, j) * 10.0 ** (-3.0 * j.astype(np.float64) / L)
    h = np.empty(L, dtype=np.float64)
    h[0] = 1.0
    h[1:] = tail / np.sqrt(np.sum(tail * tail))
    return h


def reverb(x: np.ndarray, rt60: float, seed: int) -> np.ndarray:
    return np.convolve(np.asarray(x, dtype=np.float64), rir(rt60, seed))[: len(x)]


def noise(x: np.ndarray, snr_db: float, seed: int):
    """(x + s g, s g) with s = sqrt(P_x / (P_g 10^(snr/10))), P = mean square over the clip; a silent clip passes unchanged."""
    x = np.asarray(x, dtype=np.float64)
    g = gaussian(seed, STREAM_NOISE, np.arange(len(x), dtype=np.int64))
    px, pg = np.mean(x * x), np.mean(g * g)
    if px == 0.0:
        return x.copy(), np.zeros_like(x)
    s = np.sqrt(px / (pg * 10.0 ** (float(np.float32(snr_db)) / 10.0)))
    return x + s * g, s * g


def clip_gain(gain_db: float) -> np.float32:
    return np.float32(10.0 ** (float(np.float32(gain_db)) / 20.0))


def clip(x: np.ndarray, gain_db: float) -> np.ndarray:
    """float32: clamp(x * fl32(10^(gain/20)), -1, 1)."""
    return np.clip(np.asarray(x, dtype=np.float32) * clip_gain(gain_db), np.float32(-1.0), np.float32(1.0))


def kaiser_lowpass(f: int) -> np.ndarray:
    """firwin(20 f + 1, 1 / f, window=('kaiser', 5.0)): windowed sinc, scaled to unit gain at DC."""
    numtaps = 20 * f + 1
    m = np.arange(numtaps, dtype=np.float64) - (numtaps - 1) / 2.0
    cutoff = 1.0 / f
    h = cutoff * np.sinc(cutoff * m) * np.kaiser(numtaps, 5.0)
    return h / np.sum(h)


def upfirdn_keep(h: np.ndarray, x: np.ndarray, up: int, down: int, n_keep: int) -> np.ndarray:
    """Samples [pre, pre + n_keep) of upfirdn(h', x, up, down) with h' = h * up behind the zero padding resample_poly adds:
    out[o] = sum_m up h[m] x_up[(o + pre) down - pad - m], x_up[t] = x[t / up] when up divides t."""
    half_len = (len(h) - 1) // 2
    pad = down - half_len % down
    pre = (half_len + pad) // down
    x = np.asarray(x, dtype=np.float64)
    out = np.zeros(n_keep, dtype=np.float64)
    t0 = (np.arange(n_keep, dtype=np.int64) + pre) * down - pad
    for m in range(len(h)):
        t = t0 - m
        q = t // up
        ok = (t % up == 0) & (q >= 0) & (q < len(x))
        out[ok] += (up * h[m]) * x[q[ok]]
    return out


def band(x: np.ndarray, band_rate: int) -> np.ndarray:
    """resample_poly(x, 1, f) then resample_poly(., f, 1), cut to len(x); f = 16000 / band_rate."""
    f = SR // int(band_rate)
    n = len(x)
    h = kaiser_lowpass(f)
    mid = upfirdn_keep(h, x, 1, f, -(-n // f))
    return upfirdn_keep(h, mid, f, 1, n)


_SEG_UEND = (0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF, 0x1FFF)


def lin2ulaw(s16: np.ndarray) -> np.ndarray:
    """audioop.lin2ulaw on int16 samples: the Sun G.711 encoder on the 14-bit value s >> 2."""
    v = np.asarray(s16, dtype=np.int64) >> 2
    mask = np.where(v < 0, 0x7F, 0xFF)
    v = np.minimum(np.abs(v), 8159) + (0x84 >> 2)
    seg = np.zeros_like(v)
    for e in _SEG_UEND:
        seg += v > e
    uval = np.where(seg >= 8, 0x7F, (seg << 4) | ((v >> (seg + 1)) & 0xF))
    return (uval ^ mask).astype(np.uint8)


def ulaw2lin(u: np.ndarray) -> np.ndarray:
    """audioop.ulaw2lin to int16."""
    u = ~np.asarray(u, dtype=np.int64) & 0xFF
    t = (((u & 0x0F) << 3) + 0x84) << ((u & 0x70) >> 4)
    return np.where(u & 0x80, 0x84 - t, t - 0x84).astype(np.int16)


def mulaw(x: np.ndarray) -> np.ndarray:
    """float32: int16 = clamp(rint(x * 32768), -32768, 32767), G.711 round trip, / 32768."""
    s = np.clip(np.rint(np.asarray(x, dtype=np.float32) * np.float32(32768.0)), -32768, 32767).astype(np.int16)
    return ulaw2lin(lin2ulaw(s)).astype(np.float32) / np.float32(32768.0)


def degrade(x: np.ndarray, stages: int, rt60: float = 0.0, snr_db: float = 0.0, gain_db: float = 0.0, band_rate: int = 8000,
            seed: int = 0) -> np.ndarray:
    """One variant, float64 between stages (float32 where the stage itself is stated in float32)."""
    y = np.asarray(x, dtype=np.float32).astype(np.float64)
    if stages & REVERB:
        y = reverb(y, rt60, seed)
    if stages & NOISE:
        y = noise(y, snr_db, seed)[0]
    if stages & CLIP:
        y = clip(y.astype(np.float32), gain_db).astype(np.float64)
    if stages & BAND:
        y = band(y, band_rate)
    if stages & MULAW:
        y = mulaw(y.astype(np.float32)).astype(np.float64)
    return y
