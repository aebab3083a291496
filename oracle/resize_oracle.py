"""numpy restatement of OpenCV's 8-bit down- and re-upscale of a frame:
    cv2.resize(cv2.resize(frame, (w, h), interpolation=INTER_AREA), (W, H), interpolation=INTER_LINEAR)
for a uint8 (H, W, C) frame and 1 <= h <= H, 1 <= w <= W; (h, w) == (H, W) returns the frame unchanged.  Every step is integer
or float32 arithmetic with a fixed order of operations, so it is reproduced bit for bit (tests/test_resize.py checks it against
cv2).  The GPU tests build their reference windows with this module, so they do not need cv2.

Down pass, INTER_AREA (scale = 1 / (w / W) per axis, in double):
    both ratios exactly 2:          out = (2x2 block sum + 2) >> 2
    both ratios integers (kx, ky):  out = rint(float32(block sum) * float32(1 / (kx * ky)))
    otherwise:                      per axis, source index i overlaps output cell d with weight overlap / cell width, computed in
                                    double and stored as float32 (computeResizeAreaTab); row sums accumulate S * wx in float32 in
                                    increasing column order, the output accumulates row_sum * wy in float32 in increasing row
                                    order, every product and sum rounded on its own (no fused multiply-add); out = rint, saturated.
Up pass, INTER_LINEAR (scale = 1 / (W / w) per axis, in double), fixed point with 11 fractional bits:
    f = float32((d + 0.5) * scale - 0.5), s = floor(f), f -= s, a0 = rint((1 - f) * 2048), a1 = rint(f * 2048) in float32
    columns: s < 0 -> s = 0, f = 0; s >= w - 1 -> s = w - 1, f = 0; R = a0 * S[s] + a1 * S[min(s + 1, w - 1)]  (int)
    rows: s and f are not clamped; the two rows read are clamp(s, 0, h - 1) and clamp(s + 1, 0, h - 1)
    out = (((b0 * (R0 >> 4)) >> 16) + ((b1 * (R1 >> 4)) >> 16) + 2) >> 2
rint is round half to even throughout."""
import numpy as np

COEF_BITS = 11
COEF_SCALE = 1 << COEF_BITS


def _scale(src: int, dst: int) -> float:
    return 1.0 / (float(dst) / float(src))


def area_taps(src: int, dst: int):
    """INTER_AREA's generic taps along one axis (computeResizeAreaTab): (dst index, src index, float32 weight) in the order the
    sums accumulate them."""
    scale = _scale(src, dst)
    taps = []
    for d in range(dst):
        f1 = d * scale
        f2 = f1 + scale
        cell = min(scale, src - f1)
        s1, s2 = int(np.ceil(f1)), int(np.floor(f2))
        s2 = min(s2, src - 1)
        s1 = min(s1, s2)
        if s1 - f1 > 1e-3:
            taps.append((d, s1 - 1, np.float32((s1 - f1) / cell)))
        for s in range(s1, s2):
            taps.append((d, s, np.float32(1.0 / cell)))
        if f2 - s2 > 1e-3:
            taps.append((d, s2, np.float32(min(min(f2 - s2, 1.0), cell) / cell)))
    return taps


def area_integer_ratio(src: int, dst: int) -> int:
    """The integer ratio src / dst when INTER_AREA takes its integer path on this axis (|scale - int(scale)| < DBL_EPSILON), else 0."""
    scale = _scale(src, dst)
    k = int(round(scale))
    return k if abs(scale - k) < np.finfo(np.float64).eps else 0


def linear_taps(src: int, dst: int, clamp: bool):
    """INTER_LINEAR's taps along one axis: (s0, s1, a0, a1) int64 arrays of length dst, source indices already clamped to
    0 .. src-1 for reading.  clamp: the column rule (s and f clamped at the borders); rows keep f (clamp=False)."""
    scale = _scale(src, dst)
    s0 = np.zeros(dst, np.int64)
    a = np.zeros((dst, 2), np.int64)
    for d in range(dst):
        f = np.float32((d + 0.5) * scale - 0.5)
        s = int(np.floor(f))
        f = np.float32(f - np.float32(s))
        if clamp:
            if s < 0:
                s, f = 0, np.float32(0)
            if s >= src - 1:
                s, f = src - 1, np.float32(0)
        s0[d] = s
        a[d, 0] = int(np.rint(np.float32(np.float32(1.0) - f) * np.float32(COEF_SCALE)))
        a[d, 1] = int(np.rint(f * np.float32(COEF_SCALE)))
    return np.clip(s0, 0, src - 1), np.clip(s0 + 1, 0, src - 1), a[:, 0], a[:, 1]


def downscale_area(frame: np.ndarray, h: int, w: int) -> np.ndarray:
    """cv2.resize(frame, (w, h), interpolation=cv2.INTER_AREA) for a uint8 (H, W, C) frame, h <= H, w <= W."""
    H, W = frame.shape[:2]
    if (h, w) == (H, W):
        return frame.copy()
    kx, ky = area_integer_ratio(W, w), area_integer_ratio(H, h)
    src = frame.astype(np.int64)
    if kx and ky:
        blocks = src.reshape(h, ky, w, kx, -1).sum(axis=(1, 3))
        if kx == 2 and ky == 2:
            return ((blocks + 2) >> 2).astype(np.uint8)
        prod = blocks.astype(np.float32) * np.float32(1.0 / (kx * ky))
        return np.clip(np.rint(prod), 0, 255).astype(np.uint8)
    f = frame.astype(np.float32)
    rows = np.zeros((H, w, f.shape[2]), np.float32)
    for d, s, wt in area_taps(W, w):
        rows[:, d] = rows[:, d] + f[:, s] * wt
    out = np.zeros((h, w, f.shape[2]), np.float32)
    for d, s, wt in area_taps(H, h):
        out[d] = out[d] + rows[s] * wt
    return np.clip(np.rint(out), 0, 255).astype(np.uint8)


def upscale_linear(small: np.ndarray, H: int, W: int) -> np.ndarray:
    """cv2.resize(small, (W, H), interpolation=cv2.INTER_LINEAR) for a uint8 (h, w, C) frame, h <= H, w <= W."""
    h, w = small.shape[:2]
    if (h, w) == (H, W):
        return small.copy()
    S = small.astype(np.int64)
    x0, x1, a0, a1 = linear_taps(w, W, clamp=True)
    R = S[:, x0] * a0[None, :, None] + S[:, x1] * a1[None, :, None]          # (h, W, C)
    y0, y1, b0, b1 = linear_taps(h, H, clamp=False)
    out = (((b0[:, None, None] * (R[y0] >> 4)) >> 16) + ((b1[:, None, None] * (R[y1] >> 4)) >> 16) + 2) >> 2
    return out.astype(np.uint8)


def down_up(frame: np.ndarray, h: int, w: int) -> np.ndarray:
    """One frame at face size (h, w): INTER_AREA down to (h, w), INTER_LINEAR back to the frame's size."""
    H, W = frame.shape[:2]
    assert 1 <= h <= H and 1 <= w <= W, (h, w, H, W)
    if (h, w) == (H, W):
        return frame.copy()
    return upscale_linear(downscale_area(frame, h, w), H, W)


def down_up_window(win: np.ndarray, h: int, w: int) -> np.ndarray:
    """down_up on every frame of a (T, H, W, C) window."""
    return np.stack([down_up(f, h, w) for f in win])
