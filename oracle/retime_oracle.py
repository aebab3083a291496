"""numpy restatement of a retimed window (lsd_score_retimes / lsd_retime_windows).

A variant is one row per output frame t of the window: up to 4 taps (src, weight).  src is a frame offset from the window's first
track frame; the tap reads track frame clamp(start + src, 0, n_frames - 1) (a replicate border in time: frames outside the window
but inside the track are the track's own).  Weights are Q15 integers >= 0 summing to 32768, and every byte is

    out = (sum_i weight_i * p_i + 16384) >> 15

exact integer arithmetic, so the GPU tests compare the device's bytes with this module's bit for bit."""
import numpy as np

ONE = 32768


def retime_window(track: np.ndarray, start: int, src: np.ndarray, weight: np.ndarray) -> np.ndarray:
    """Window [start, start + T) of a uint8 (n_frames, H, W, C) track retimed by (src, weight) of shape (T, n): (T, H, W, C) uint8."""
    src = np.asarray(src, np.int64)
    weight = np.asarray(weight, np.int64)
    assert src.shape == weight.shape and src.ndim == 2, (src.shape, weight.shape)
    assert (weight >= 0).all() and (weight.sum(axis=1) == ONE).all()
    frames = np.clip(int(start) + src, 0, track.shape[0] - 1)
    acc = np.full((src.shape[0],) + track.shape[1:], ONE // 2, np.int64)
    for i in range(src.shape[1]):
        acc += weight[:, i, None, None, None] * track[frames[:, i]].astype(np.int64)
    return (acc >> 15).astype(np.uint8)
