"""numpy restatement of OpenCV's baseline JPEG encode followed by decode (libjpeg-turbo, JDCT_ISLOW):
    cv2.imdecode(cv2.imencode('.jpg', bgr, [IMWRITE_JPEG_QUALITY, q (, IMWRITE_JPEG_SAMPLING_FACTOR, 444)]), IMREAD_COLOR)
for a uint8 (H, W, 3) frame whose sides are multiples of the MCU (16 for 4:2:0, 8 for 4:4:4).  Entropy coding is lossless, so the
round trip is integer arithmetic from pixels to pixels and is reproduced bit for bit (tests/test_jpeg.py checks it against cv2):
    RGB -> YCbCr (jccolor.c), 4:2:0: 2x2 box downsampling with alternating bias 1, 2 (jcsample.c h2v2_downsample),
    per 8x8 block: level shift, jfdctint, quantisation by 8 * qtab with rounding, dequantisation, jidctint with its range limit,
    4:2:0: fancy upsampling (jdsample.c h2v2_fancy_upsample), YCbCr -> RGB (jdcolor.c).
Every intermediate is checked to fit in int32: the CUDA kernel (csrc/jpeg.cu) computes in int32.  The GPU tests build their
reference windows with this module, so they do not need cv2."""
import numpy as np

CONST_BITS, PASS1_BITS = 13, 2
F0298, F0390, F0541, F0765, F0899, F1175 = 2446, 3196, 4433, 6270, 7373, 9633
F1501, F1847, F1961, F2053, F2562, F3072 = 12299, 15137, 16069, 16819, 20995, 25172
I32_MIN, I32_MAX = -(1 << 31), (1 << 31) - 1

# IJG Annex K tables, natural (row-major) order
LUMA = np.array([16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
                 14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
                 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99], dtype=np.int64).reshape(8, 8)
CHROMA = np.array([17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99,
                   47, 66, 99, 99, 99, 99, 99, 99] + [99] * 32, dtype=np.int64).reshape(8, 8)


def fix(x: float) -> int:
    return int(x * 65536 + 0.5)


def _i32(*arrays):
    for a in arrays:
        a = np.asarray(a)
        assert a.size == 0 or (a.min() >= I32_MIN and a.max() <= I32_MAX), "intermediate outside int32"
    return arrays[0] if len(arrays) == 1 else arrays


def _descale(x, n):
    return _i32(x + (1 << (n - 1))) >> n


def quality_table(base, quality: int) -> np.ndarray:
    """jpeg_quality_scaling + jpeg_add_quant_table with force_baseline: (8, 8) int64 in natural order."""
    q = max(1, min(100, int(quality)))
    s = 5000 // q if q < 50 else 200 - 2 * q
    return np.clip((np.asarray(base, dtype=np.int64) * s + 50) // 100, 1, 255)


def fdct_1d(d, pass_: int):
    """jfdctint along the last axis; pass 0 is the row pass, 1 the column pass."""
    d = [d[..., i] for i in range(8)]
    t0, t7, t1, t6 = d[0] + d[7], d[0] - d[7], d[1] + d[6], d[1] - d[6]
    t2, t5, t3, t4 = d[2] + d[5], d[2] - d[5], d[3] + d[4], d[3] - d[4]
    t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    o = [None] * 8
    if pass_ == 0:
        o[0], o[4], sh = (t10 + t11) << PASS1_BITS, (t10 - t11) << PASS1_BITS, CONST_BITS - PASS1_BITS
    else:
        o[0], o[4], sh = _descale(t10 + t11, PASS1_BITS), _descale(t10 - t11, PASS1_BITS), CONST_BITS + PASS1_BITS
    z1 = _i32((t12 + t13) * F0541)
    o[2] = _descale(z1 + _i32(t13 * F0765), sh)
    o[6] = _descale(z1 - _i32(t12 * F1847), sh)
    z1, z2, z3, z4 = t4 + t7, t5 + t6, t4 + t6, t5 + t7
    z5 = _i32((z3 + z4) * F1175)
    t4, t5, t6, t7 = _i32(t4 * F0298, t5 * F2053, t6 * F3072, t7 * F1501)
    z1, z2 = _i32(z1 * -F0899, z2 * -F2562)
    z3, z4 = _i32(z3 * -F1961 + z5, z4 * -F0390 + z5)
    o[7], o[5] = _descale(t4 + z1 + z3, sh), _descale(t5 + z2 + z4, sh)
    o[3], o[1] = _descale(t6 + z2 + z3, sh), _descale(t7 + z1 + z4, sh)
    return _i32(np.stack(o, -1))


def idct_1d(c, pass_: int):
    """jidctint along the last axis; pass 0 is the column pass, 1 the row pass (before the range limit)."""
    c = [c[..., i] for i in range(8)]
    z2, z3 = c[2], c[6]
    z1 = _i32((z2 + z3) * F0541)
    t2, t3 = _i32(z1 - z3 * F1847, z1 + z2 * F0765)
    t0, t1 = _i32((c[0] + c[4]) << CONST_BITS, (c[0] - c[4]) << CONST_BITS)
    t10, t13, t11, t12 = _i32(t0 + t3, t0 - t3, t1 + t2, t1 - t2)
    a0, a1, a2, a3 = c[7], c[5], c[3], c[1]
    z1, z2, z3, z4 = a0 + a3, a1 + a2, a0 + a2, a1 + a3
    z5 = _i32((z3 + z4) * F1175)
    a0, a1, a2, a3 = _i32(a0 * F0298, a1 * F2053, a2 * F3072, a3 * F1501)
    z1, z2 = _i32(z1 * -F0899, z2 * -F2562)
    z3, z4 = _i32(z3 * -F1961 + z5, z4 * -F0390 + z5)
    a0, a1, a2, a3 = _i32(a0 + z1 + z3, a1 + z2 + z4, a2 + z2 + z3, a3 + z1 + z4)
    sh = CONST_BITS + PASS1_BITS + 3 if pass_ == 1 else CONST_BITS - PASS1_BITS
    o = [t10 + a3, t11 + a2, t12 + a1, t13 + a0, t13 - a0, t12 - a1, t11 - a2, t10 - a3]
    return np.stack([_descale(v, sh) for v in o], -1)


def range_limit(x):
    """jidctint's sample range limit of a descaled output x (centred on 0) -> 0..255."""
    m = x & 1023
    return np.where(m < 128, m + 128, np.where(m < 512, 255, np.where(m < 896, 0, m - 896)))


def plane_round_trip(P, qtab):
    """One component plane (h, w) of samples 0..255, both multiples of 8: DCT, quantise, dequantise, inverse DCT."""
    h, w = P.shape
    blk = (P - 128).reshape(h // 8, 8, w // 8, 8).transpose(0, 2, 1, 3)        # (by, bx, row, col)
    c = fdct_1d(blk, 0)
    c = fdct_1d(c.swapaxes(-1, -2), 1).swapaxes(-1, -2)
    d = qtab * 8
    qc = np.sign(c) * ((np.abs(c) + (d >> 1)) // d)
    x = idct_1d(_i32(qc * qtab).swapaxes(-1, -2), 0).swapaxes(-1, -2)
    x = idct_1d(x, 1)
    return range_limit(x).transpose(0, 2, 1, 3).reshape(h, w)


def downsample_h2v2(P):
    s = P[0::2, 0::2] + P[0::2, 1::2] + P[1::2, 0::2] + P[1::2, 1::2]
    bias = np.where(np.arange(s.shape[1]) % 2 == 0, 1, 2)
    return (s + bias) >> 2


def upsample_h2v2_fancy(P):
    h, w = P.shape
    above = np.vstack([P[:1], P[:-1]])
    below = np.vstack([P[1:], P[-1:]])
    out = np.zeros((2 * h, 2 * w), dtype=np.int64)
    for r, far in ((0, above), (1, below)):
        cs = 3 * P + far
        left = np.hstack([cs[:, :1], cs[:, :-1]])
        right = np.hstack([cs[:, 1:], cs[:, -1:]])
        even = (3 * cs + left + 8) >> 4
        odd = (3 * cs + right + 7) >> 4
        even[:, 0] = (4 * cs[:, 0] + 8) >> 4
        odd[:, -1] = (4 * cs[:, -1] + 7) >> 4
        out[r::2, 0::2] = even
        out[r::2, 1::2] = odd
    return out


def round_trip_bgr(bgr: np.ndarray, quality: int, sampling: str = "420") -> np.ndarray:
    """cv2.imdecode(cv2.imencode('.jpg', bgr, quality, sampling)) of a uint8 (H, W, 3) BGR frame."""
    if sampling not in ("420", "444"):
        raise ValueError(f"sampling must be '420' or '444', got {sampling!r}")
    H, W = bgr.shape[:2]
    mcu = 16 if sampling == "420" else 8
    if H % mcu or W % mcu:
        raise ValueError(f"{H}x{W} frame: sides must be multiples of {mcu} for {sampling}")
    b, g, r = (bgr[..., i].astype(np.int64) for i in range(3))
    half = 1 << 15
    Y = (fix(.299) * r + fix(.587) * g + fix(.114) * b + half) >> 16
    Cb = (-fix(.16874) * r - fix(.33126) * g + fix(.5) * b + (128 << 16) + half - 1) >> 16
    Cr = (fix(.5) * r - fix(.41869) * g - fix(.08131) * b + (128 << 16) + half - 1) >> 16
    ql, qc = quality_table(LUMA, quality), quality_table(CHROMA, quality)
    y = plane_round_trip(Y, ql)
    if sampling == "420":
        cb = upsample_h2v2_fancy(plane_round_trip(downsample_h2v2(Cb), qc))
        cr = upsample_h2v2_fancy(plane_round_trip(downsample_h2v2(Cr), qc))
    else:
        cb, cr = plane_round_trip(Cb, qc), plane_round_trip(Cr, qc)
    x, z = cr - 128, cb - 128
    R = y + ((fix(1.402) * x + half) >> 16)
    B = y + ((fix(1.772) * z + half) >> 16)
    G = y + ((-fix(.34414) * z - fix(.71414) * x + half) >> 16)
    return np.stack([np.clip(v, 0, 255) for v in (B, G, R)], -1).astype(np.uint8)


def round_trip(frame: np.ndarray, quality: int, sampling, channel_order: str = "rgb") -> np.ndarray:
    """The round trip of a frame in `channel_order` ("rgb" or "bgr"); sampling None returns the frame unchanged.  For an RGB
    frame this is cvtColor(imdecode(imencode(cvtColor(frame, RGB2BGR))), BGR2RGB)."""
    if sampling is None:
        return frame.copy()
    if channel_order == "bgr":
        return round_trip_bgr(frame, quality, sampling)
    if channel_order != "rgb":
        raise ValueError(f"channel_order must be 'rgb' or 'bgr', got {channel_order!r}")
    return round_trip_bgr(frame[..., ::-1], quality, sampling)[..., ::-1]


def round_trip_window(win: np.ndarray, quality: int, sampling, channel_order: str = "rgb") -> np.ndarray:
    """A uint8 window (T, H, W, 3), every frame round-tripped."""
    return np.stack([round_trip(win[t], quality, sampling, channel_order) for t in range(win.shape[0])])
