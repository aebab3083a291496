"""numpy restatement of OpenCV's 8-bit bilinear affine warp with replicated borders:
    cv2.warpAffine(src, M, (W, H), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)
for a uint8 (H, W, C) image and a forward 2x3 matrix M (src -> dst).  Once its per-row and per-column terms are tabulated the
warp is integer arithmetic, so it is reproduced bit for bit (tests/test_warps.py checks it against cv2).  The GPU tests build
their reference windows with it, so they do not need cv2.

    Minv = invert(M)                                           (cv::warpAffine's own inversion order, in double)
    adelta[x] = rint(Minv[0,0]*x*1024)                         bdelta[x] = rint(Minv[1,0]*x*1024)        rint: half to even
    X0[y] = rint((Minv[0,1]*y + Minv[0,2])*1024) + 16          Y0[y] = rint((Minv[1,1]*y + Minv[1,2])*1024) + 16
    X = (X0[y] + adelta[x]) >> 5,  Y = (Y0[y] + bdelta[x]) >> 5
    xi = X >> 5, fx = X & 31, yi = Y >> 5, fy = Y & 31
    out = clamp((sum_k TAB[fy,fx,k] * src[clamp(yi+dy_k), clamp(xi+dx_k), c] + 16384) >> 15, 0, 255)
"""
import numpy as np

AB_BITS, INTER_BITS, COEF_BITS = 10, 5, 15
AB_SCALE, INTER_TAB, COEF_SCALE = 1 << AB_BITS, 1 << INTER_BITS, 1 << COEF_BITS
TAPS = ((0, 0), (0, 1), (1, 0), (1, 1))          # (dy, dx) of the four weights


def invert_affine(M) -> np.ndarray:
    """The inverse cv::warpAffine takes when WARP_INVERSE_MAP is not set, in its order of operations (no fused multiply-add)."""
    m0, m1, m2, m3, m4, m5 = (float(v) for v in np.asarray(M, dtype=np.float64).reshape(6))
    D = m0 * m4 - m1 * m3
    D = 1.0 / D if D != 0.0 else 0.0
    a0, a1 = m4 * D, -m1 * D
    a3, a4 = -m3 * D, m0 * D
    a2 = -a0 * m2 - a1 * m5
    a5 = -a3 * m2 - a4 * m5
    return np.array([[a0, a1, a2], [a3, a4, a5]], dtype=np.float64)


def weight_table() -> np.ndarray:
    """(32, 32, 4) int64: cv2's bilinear table (initInterTab2D), weights rint(w * 32768) whose sum is fixed to 32768 (a deficit
    goes to the largest weight, an excess comes off the smallest).  For bilinear weights every product is exact, so no fix is
    ever needed and TAB[fy, fx] = 32 * ((32-fy)(32-fx), (32-fy) fx, fy (32-fx), fy fx) (pinned by the tests)."""
    t = np.zeros((INTER_TAB, INTER_TAB, 4), dtype=np.int64)
    for i in range(INTER_TAB):
        for j in range(INTER_TAB):
            fy, fx = i / INTER_TAB, j / INTER_TAB
            w = np.array([(1 - fy) * (1 - fx), (1 - fy) * fx, fy * (1 - fx), fy * fx])
            iw = np.rint(w * COEF_SCALE).astype(np.int64)
            s = int(iw.sum())
            if s != COEF_SCALE:
                k = int(np.argmax(iw)) if s < COEF_SCALE else int(np.argmin(iw))
                iw[k] += COEF_SCALE - s
            t[i, j] = iw
    return t


TAB = weight_table()


def warp_tables(M, H: int, W: int):
    """(X0 (H,), Y0 (H,), adelta (W,), bdelta (W,)) int64: the per-row and per-column terms of the warp of an H x W frame."""
    A = invert_affine(M)
    xs, ys = np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64)
    adelta = np.rint(A[0, 0] * xs * AB_SCALE).astype(np.int64)
    bdelta = np.rint(A[1, 0] * xs * AB_SCALE).astype(np.int64)
    rd = AB_SCALE // INTER_TAB // 2
    X0 = np.rint((A[0, 1] * ys + A[0, 2]) * AB_SCALE).astype(np.int64) + rd
    Y0 = np.rint((A[1, 1] * ys + A[1, 2]) * AB_SCALE).astype(np.int64) + rd
    return X0, Y0, adelta, bdelta


def warp_affine(src: np.ndarray, M) -> np.ndarray:
    """cv2.warpAffine(src, M, (W, H), flags=INTER_LINEAR, borderMode=BORDER_REPLICATE) of a uint8 (H, W, C) image."""
    H, W, C = src.shape
    X0, Y0, adelta, bdelta = warp_tables(M, H, W)
    sh = AB_BITS - INTER_BITS
    X = (X0[:, None] + adelta[None, :]) >> sh
    Y = (Y0[:, None] + bdelta[None, :]) >> sh
    xi, fx = X >> INTER_BITS, X & (INTER_TAB - 1)
    yi, fy = Y >> INTER_BITS, Y & (INTER_TAB - 1)
    w = TAB[fy, fx]                                                  # (H, W, 4)
    acc = np.zeros((H, W, C), dtype=np.int64)
    for k, (dy, dx) in enumerate(TAPS):
        yy = np.clip(yi + dy, 0, H - 1)
        xx = np.clip(xi + dx, 0, W - 1)
        acc += w[:, :, k:k + 1] * src[yy, xx].astype(np.int64)
    return np.clip((acc + (1 << (COEF_BITS - 1))) >> COEF_BITS, 0, 255).astype(np.uint8)


def warp_window(win: np.ndarray, mats) -> np.ndarray:
    """A uint8 window (T, H, W, 3) with frame t warped by mats[t] (a (T, 2, 3) array, or one (2, 3) matrix for every frame)."""
    mats = np.asarray(mats, dtype=np.float64)
    if mats.ndim == 2:
        mats = np.broadcast_to(mats, (win.shape[0], 2, 3))
    return np.stack([warp_affine(win[t], mats[t]) for t in range(win.shape[0])])
