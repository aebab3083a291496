"""Temporal robustness: the retime table builders of `Predictor`, `Predictor.score_track_retimes` (lsd_score_retimes),
`Predictor.retime_track_windows` (lsd_retime_windows), `Predictor.temporal_track` and the `temporal` entry of
`predict_long_video_from_tracks`.  Every output byte is (sum w_i p_i + 16384) >> 15 over taps clamped to the track:
oracle/retime_oracle.py restates it, and the logit of (window, variant) must be bit for bit the plain forward's logit for that
window retimed on the host by the oracle."""
import ctypes as C
import json
from fractions import Fraction

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import augmentation_stability, lowest_stable_quality
from oracle import retime_oracle as rto
from tests.golden.long_video_synth import SCENARIOS, make_audio, make_tracks

P = lb.Predictor
ONE = 32768
NAMES_15 = ["none", "hold12", "hold10", "hold8", "hold6", "hold5", "blend10", "freeze4", "freeze10", "loss10", "drift8", "exposure3"]
RATES_15 = [None, 12, 10, 8, 6, 5, None, None, None, None, None, None]


def _one_tap(tab):
    """The src column of a table whose every frame is one full-weight tap."""
    src, wt = tab
    assert src.shape == wt.shape == (len(src), 4) and src.dtype == wt.dtype == np.int32
    assert (wt[:, 0] == ONE).all() and (wt[:, 1:] == 0).all()
    return src[:, 0].tolist()


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_hold_retime_hand_computed():
    assert _one_tap(P.hold_retime(32, 15, 5)) == [3 * (t // 3) for t in range(32)]
    # captures at frames 1.5 and 4.5 round up to 2 and 5
    assert _one_tap(P.hold_retime(32, 15, 10))[:9] == [0, 0, 2, 3, 3, 5, 6, 6, 8]
    assert _one_tap(P.hold_retime(32, 15, 15)) == list(range(32))
    assert _one_tap(P.hold_retime(8, 15, 30)) == list(range(8))


@pytest.mark.parametrize("fps", [10, 12, 25, 30, 30000 / 1001])
def test_hold_retime_matches_float64(fps):
    """Every hold rate below the video's rate (a source of rate == fps is the plain window, where float64 rounds 9 * r / r below 9
    for NTSC rates and the exact rationals do not)."""
    for rate in [r for r in (5, 6, 8, 10, 12, 15, 24, 25) if r < fps]:
        want = [int(np.floor(np.floor(t * rate / fps) * fps / rate + 0.5)) for t in range(64)]
        got = _one_tap(P.hold_retime(64, fps, rate))
        assert got == want, (fps, rate)
        assert all(s <= t for t, s in enumerate(got))


def test_exact_rates():
    assert P._exact_rate(30000 / 1001, "fps") == Fraction(30000, 1001)
    assert P._exact_rate(29.97, "fps") == Fraction(2997, 100)
    assert P._exact_rate(15.0, "fps") == 15
    with pytest.raises(ValueError):
        P._exact_rate(0, "fps")


def test_blend_retime_hand_computed():
    src, wt = P.blend_retime(6, 15, 10)
    assert src[0].tolist() == [0, 0, 0, 0] and wt[0].tolist() == [ONE, 0, 0, 0]
    assert src[1, :2].tolist() == [0, 2] and wt[1].tolist() == [ONE - 21845, 21845, 0, 0]        # 2/3 of the way to capture 1
    assert src[2, :2].tolist() == [2, 3] and wt[2].tolist() == [ONE - 10923, 10923, 0, 0]        # 1/3 of the way to capture 2
    assert src[3, 0] == 3 and wt[3].tolist() == [ONE, 0, 0, 0]
    assert (wt.sum(axis=1) == ONE).all()
    # at the frame rate itself every frame is one tap: the plain window
    assert _one_tap(P.blend_retime(16, 15, 15)) == list(range(16))


def test_freeze_and_drop_hand_computed():
    assert _one_tap(P.freeze_retime(8, 3, 2)) == [0, 1, 2, 2, 2, 5, 6, 7]
    assert _one_tap(P.freeze_retime(8, 0, 2)) == [-1, -1, 2, 3, 4, 5, 6, 7]             # before the window: clamped to the track
    assert _one_tap(P.freeze_retime(32, 16, 10)) == list(range(16)) + [15] * 10 + list(range(26, 32))
    assert _one_tap(P.drop_retime(10, 4, repeat=True)) == [0, 1, 2, 2, 4, 5, 6, 6, 8, 9]
    assert _one_tap(P.drop_retime(10, 4, repeat=False)) == [0, 1, 2, 4, 5, 6, 8, 9, 10, 12]
    drift = _one_tap(P.drop_retime(32, 8, repeat=False))
    assert drift[31] - 31 == 4                                                            # 4 frames ahead by the last frame
    with pytest.raises(ValueError):
        P.drop_retime(32, 1)
    with pytest.raises(ValueError):
        P.freeze_retime(32, -1, 2)


@pytest.mark.parametrize("n", [2, 3, 4])
def test_exposure_retime(n):
    src, wt = P.exposure_retime(32, n)
    c = (n - 1) // 2
    assert (wt.sum(axis=1) == ONE).all()
    for t in range(32):
        assert src[t, :n].tolist() == [t - c + i for i in range(n)]
        assert wt[t, :n].tolist() == [ONE // n + (ONE % n if i == c else 0) for i in range(n)]
        assert (wt[t, n:] == 0).all()
    if n == 3:
        assert wt[0, :3].tolist() == [10922, 10924, 10922]
    with pytest.raises(ValueError):
        P.exposure_retime(32, 5)


def test_loss_retime():
    a = _one_tap(P.loss_retime(32, 0.10, 3, seed=0))
    assert a == _one_tap(P.loss_retime(32, 0.10, 3, seed=0))
    assert a[0] == 0 and all(s <= t for t, s in enumerate(a)) and a == sorted(a)
    # a restatement of the Gilbert-Elliott chain: one draw per frame from frame 1 on
    g = np.random.default_rng(0)
    good, last, want = True, 0, [0]
    for t in range(1, 32):
        u = g.random()
        good = u >= 0.10 / (3 * 0.9) if good else u < 1 / 3
        last = t if good else last
        want.append(last)
    assert a == want
    assert _one_tap(P.loss_retime(32, 0.0, 3, seed=5)) == list(range(32))
    long = _one_tap(P.loss_retime(20000, 0.10, 3, seed=1))
    lost = sum(1 for t, s in enumerate(long) if s != t)
    assert 0.08 < lost / 20000 < 0.12
    assert _one_tap(P.loss_retime(32, 0.10, 3, seed=1)) != a
    for bad in ((1.0, 3), (-0.1, 3), (0.1, 0.5), (0.9, 1)):
        with pytest.raises(ValueError):
            P.loss_retime(32, *bad)


def test_builder_range_check():
    assert _one_tap(P.hold_retime(32, 15, 0.2)) == [0] * 32                 # a capture every 75 frames: the first one held
    with pytest.raises(ValueError):
        P.blend_retime(32, 15, 0.2)                    # ... and blending towards the next one reads frame 75, past 2T-1
    with pytest.raises(ValueError):
        P.blend_retime(32, 15, -1)


def test_default_temporal_variants():
    names, tabs, rates = P.temporal_variants(32)
    assert names == NAMES_15 and rates == RATES_15 and len(tabs) == 12
    assert _one_tap(tabs[0]) == list(range(32))
    assert _one_tap(tabs[1]) == _one_tap(P.hold_retime(32, 15, 12))
    assert _one_tap(tabs[NAMES_15.index("freeze4")]) == _one_tap(P.freeze_retime(32, 16, 4))
    assert _one_tap(tabs[NAMES_15.index("drift8")]) == _one_tap(P.drop_retime(32, 8, repeat=False))
    assert all(np.array_equal(a, b) for a, b in zip(tabs[6], P.blend_retime(32, 15, 10)))
    assert all(np.array_equal(a, b) for a, b in zip(tabs[9], P.loss_retime(32, 0.10, 3, 0)))
    assert all(np.array_equal(a, b) for a, b in zip(tabs[11], P.exposure_retime(32, 3)))
    names, tabs, rates = P.temporal_variants(32, fps=10)
    assert names == ["none", "hold8", "hold6", "hold5", "freeze4", "freeze10", "loss10", "drift8", "exposure3"]
    assert rates == [None, 8, 6, 5, None, None, None, None, None] and len(tabs) == 9
    names, _, rates = P.temporal_variants(32, fps=30000 / 1001)
    assert names == NAMES_15 and rates == RATES_15


def test_lowest_stable_fps_hand_built(monkeypatch):
    """temporal_track's report from hand-built logits (the same logit in every window of a column)."""
    pred = P(None, device=torch.device("cpu"))
    track = torch.zeros((40, 96, 96, 3), dtype=torch.uint8)
    mel = torch.zeros((1, 80, 200))

    def run(cols, **kw):
        monkeypatch.setattr(pred, "score_track_retimes", lambda *a, **k: torch.tensor([cols] * 3, dtype=torch.float32))
        return pred.temporal_track(track, [0, 4, 8], mel, 40, confidence_threshold=0.5, **kw)

    #          none hold12 hold10 hold8 hold6 hold5 blend10 freeze4 freeze10 loss10 drift8 exposure3
    res = run([4.0, 3.0, 3.0, 2.0, 1.0, 0.5, 2.0, 2.0, 2.0, 2.0, 2.0, 2.0])
    assert res["lowest_stable_fps"] == 5 and res["verdict_stable"]
    assert res["variants"] == NAMES_15 and res["rates"] == RATES_15 and res["window_starts"] == [0, 4, 8]
    assert run([4.0, 3.0, 3.0, -2.0, 1.0, 0.5, 2.0, 2.0, 2.0, 2.0, 2.0, 2.0])["lowest_stable_fps"] == 10     # flips at 8
    assert run([4.0, -3.0, 3.0, 2.0, 1.0, 0.5, 2.0, 2.0, 2.0, 2.0, 2.0, 2.0])["lowest_stable_fps"] is None   # 12 fps flips
    cols = [-3.0, -3.0, -2.0, -1.0, -0.5, -0.1, -1.0, -1.0, 0.4, -1.0, -1.0, -1.0]                        # fake; freeze10 flips
    res = run(cols, audio_starts_from=[100, 104, 108])
    assert res["lowest_stable_fps"] == 5 and not res["verdict_stable"] and res["window_starts"] == [100, 104, 108]
    probs = np.array([[pred._calibrate(x) for x in cols]] * 3)
    want = augmentation_stability(probs, 0.5, pred.confidence_smoothing, pred.trim_ratio)
    for k, v in want.items():
        assert np.array_equal(np.asarray(res[k]), np.asarray(v)), k
    assert res["lowest_stable_fps"] == lowest_stable_quality(RATES_15, want["variant_confidence"], want["confidence"], 0.5)


def _tab(src, wt):
    return np.asarray(src, np.int32), np.asarray(wt, np.int32)


T32 = np.arange(32)
GOOD = _tab(np.stack([T32, T32 + 1], 1), np.full((32, 2), ONE // 2))
BAD_VARIANTS = [
    [],                                                                   # K = 0
    [T32] * 65,                                                           # K = 65
    [np.arange(31)],                                                      # T - 1 frames
    [T32.reshape(4, 8)],                                                  # not (T,)
    [T32.astype(np.float32)],                                             # not integers
    [T32 - 33],                                                           # src below -T
    [T32 + 33],                                                           # src past 2T - 1
    [_tab(np.stack([T32, T32 + 40], 1), np.stack([np.full(32, ONE), np.zeros(32)], 1))],   # a weight-0 tap past 2T - 1
    [_tab(np.stack([T32, T32], 1), np.stack([np.full(32, ONE + 1), np.full(32, -1)], 1))],  # a negative weight
    [_tab(np.stack([T32, T32], 1), np.full((32, 2), ONE // 2 - 1))],      # weights sum to 32766
    [_tab(np.tile(T32[:, None], (1, 5)), np.full((32, 5), 0).astype(np.int32))],            # five taps
    [(GOOD[0], GOOD[1][:, :1])],                                          # src and weight shapes differ
    [(GOOD[0], GOOD[1].astype(np.float64))],                              # float weights
]


@pytest.mark.parametrize("variants", BAD_VARIANTS, ids=range(len(BAD_VARIANTS)))
def test_argument_errors_raise_value_error(variants):
    pred = P(None, device=torch.device("cpu"))
    track = torch.zeros((40, 96, 96, 3), dtype=torch.uint8)
    mel = torch.zeros((1, 80, 200))
    with pytest.raises(ValueError):
        pred.score_track_retimes(track, [0], mel, 40, variants)
    with pytest.raises(ValueError):
        pred.retime_track_windows(track, [0], variants)


def test_argument_errors_track_window_and_audio():
    pred = P(None, device=torch.device("cpu"))
    track = torch.zeros((40, 96, 96, 3), dtype=torch.uint8)
    mel = torch.zeros((1, 80, 200))
    with pytest.raises(ValueError):
        pred.retime_track_windows(track, [9], [T32])                       # window [9, 41) outside the 40-frame track
    with pytest.raises(ValueError):
        pred.retime_track_windows(track, [-1], [T32])
    with pytest.raises(ValueError):
        pred.retime_track_windows(track.float(), [0], [T32])
    with pytest.raises(ValueError):
        pred.retime_track_windows(track[..., :2], [0], [T32])
    with pytest.raises(ValueError):
        pred.score_track_retimes(track, [0], mel[0], 40, [T32])
    with pytest.raises(ValueError):
        pred.score_track_retimes(track, [0, 4], mel, 40, [T32], audio_starts_from=[0])
    # accepted forms: a bare src array or list, (src, weight) of 1 to 4 taps, every default table
    K, vc = pred._retime_args(track, [0, 8], [T32, list(range(32)), GOOD, P.exposure_retime(32, 4)] + P.temporal_variants(32)[1])
    assert K == 16 and len(vc) == 16 * 32
    assert list(vc[32 + 1].src) == [1, 0, 0, 0] and list(vc[32 + 1].weight) == [ONE, 0, 0, 0]
    assert list(vc[2 * 32 + 5].src) == [5, 6, 0, 0] and list(vc[2 * 32 + 5].weight) == [ONE // 2, ONE // 2, 0, 0]


def test_oracle_rule():
    """The oracle's rule on a hand-sized track: clamped taps and the rounding of the Q15 blend."""
    track = np.zeros((5, 1, 1, 3), np.uint8)
    track[:, 0, 0, 0] = [10, 20, 30, 40, 255]
    track[:, 0, 0, 1] = [1, 2, 3, 4, 5]
    out = rto.retime_window(track, 1, [[-3, 0], [9, 0], [0, 1], [0, 3]], [[ONE, 0], [ONE, 0], [ONE // 2, ONE // 2], [ONE - 1, 1]])
    assert out[:, 0, 0, 0].tolist() == [10, 255, 25, 20]                 # frame -2 -> 0, frame 10 -> 4, (20 + 30) / 2
    assert out[:, 0, 0, 1].tolist() == [1, 5, 3, 2]                      # (2 + 3) / 2 = 2.5 rounds half up


def test_long_video_temporal_entry():
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def temporal_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"confidence": 0.7, "lowest_stable_fps": 8, "window_starts": [int(s) for s in tr["chunk_starts"]]}

    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, temporal=True, temporal_fn=temporal_fn, **fns)
    assert "temporal" not in base
    assert set(res) == set(base) | {"temporal"}
    assert res["temporal"]["track_id"] == res["selected_track_id"] == seen[0] and len(seen) == 1
    assert res["temporal"]["lowest_stable_fps"] == 8
    tr = next(t for t in tracks if int(t["track_id"]) == seen[0])
    assert res["temporal"]["window_starts"] == [int(s) for s in tr["chunk_starts"]]
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k


def _as_chunks(tr, keep=None):
    """The same track in the reference's chunk format: (3, T, H, W) float32 = u8 / 255 windows cut at `chunk_starts` (only the
    windows in `keep` when given)."""
    crops, a = tr["crops_u8"], int(tr["track_start_frame"])
    starts = [int(s) for i, s in enumerate(tr["chunk_starts"]) if keep is None or i in keep]
    out = {k: v for k, v in tr.items() if k != "crops_u8"}
    out["chunk_starts"] = starts
    out["chunks"] = [np.ascontiguousarray(crops[s - a: s - a + 32].transpose(3, 0, 1, 2)).astype(np.float32) / np.float32(255.0)
                     for s in starts]
    return out


def test_chunk_runs_rebuild_consecutive_frames():
    """Overlapping and touching reference windows share one run of the video's own frames; a gap starts a new run."""
    from lipsync_b200.long_video import _chunk_runs
    g = np.random.default_rng(4)
    crops = g.integers(0, 256, (150, 8, 6, 3), dtype=np.uint8)
    tr = {"crops_u8": crops, "track_start_frame": 10, "chunk_starts": [10, 18, 26, 58, 100, 104, 91]}
    ch = _as_chunks(tr)
    ch["chunks"] = [c[:, :, :8, :6] for c in ch["chunks"]]
    runs = _chunk_runs(ch)
    # 10, 18, 26 overlap and 58 touches [10, 58); frame 90 is covered by no window, so 91 starts a run that 100 and 104 overlap
    assert [(first, idx) for _, first, idx in runs] == [(10, [0, 1, 2, 3]), (91, [6, 4, 5])]
    assert [c.shape[0] for c, _, _ in runs] == [80, 45]
    for c, first, _ in runs:
        assert c.dtype == torch.uint8 and np.array_equal(c.numpy(), crops[first - 10: first - 10 + c.shape[0]])


def test_long_video_temporal_chunks_scored_per_run(monkeypatch):
    """With reference-format chunks the default temporal hook scores every run of consecutive frames as its own track, with the
    windows' local starts in the run and their absolute audio starts, and reports the windows in their given order."""
    spec = SCENARIOS["one_track_localised_fake"]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    tr = tracks[0]
    keep = [i for i in range(len(tr["chunk_starts"])) if not 10 <= i <= 14]          # windows 10 .. 14 missing: frames 104 .. 119
    ch = _as_chunks(tr, keep)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    calls = []

    def score(track, starts, mel_full, total_v, variants, audio_starts_from=None):
        calls.append((track.numpy(), list(starts), list(audio_starts_from)))
        return torch.tensor([[float(a) / 100.0 - 1.0] * len(variants) for a in audio_starts_from])

    monkeypatch.setattr(pred, "score_track_retimes", score)
    fns = dict(score_fn=lambda t: [0.7] * len(t["chunk_starts"]), speech_fn=lambda t, idxs: [0.6] * len(idxs),
               mouth_fn=lambda t: {"check_result": "no_data"})
    res = lb.predict_long_video_from_tracks(pred, [ch], mel, vad, spec["fps"], n_frames, temporal=True, **fns)["temporal"]
    starts = ch["chunk_starts"]
    assert len(calls) == 2
    for track, local, absolute in calls:
        first = absolute[0] - local[0]
        assert [first + s for s in local] == absolute
        assert np.array_equal(track, tr["crops_u8"][first: first + track.shape[0]])
        assert absolute[-1] + 32 == first + track.shape[0]
    assert calls[0][2] + calls[1][2] == starts and calls[1][2][0] - (calls[0][2][-1] + 32) == 16
    names, _, rates = P.temporal_variants(32, spec["fps"])
    logits = np.array([[s / 100.0 - 1.0] * len(names) for s in starts], np.float32)
    want = pred._temporal_report(logits, names, rates, 0.5, starts)
    assert json.dumps(res, sort_keys=True, default=str) == json.dumps(dict(want, track_id=0), sort_keys=True, default=str)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()


@pytest.fixture(scope="module")
def model(built, seed0_sd):
    m = lb.LipSyncModel()
    m.load_state_dict(seed0_sd, strict=True)
    return m.to("cuda:0").eval()


def _random_taps(T, K, seed):
    """K tables of 1 to 4 taps with random weights (some taps of weight 0) anywhere in -T .. 2T-1."""
    g = np.random.default_rng(seed)
    out = []
    for _ in range(K):
        n = int(g.integers(1, 5))
        src = g.integers(-T, 2 * T, (T, n)).astype(np.int32)
        cuts = np.sort(g.integers(0, ONE + 1, (T, n - 1)), axis=1)
        wt = np.diff(np.concatenate([np.zeros((T, 1), np.int64), cuts, np.full((T, 1), ONE)], axis=1), axis=1).astype(np.int32)
        out.append((src, wt))
    return out


def _edge_taps(T):
    """Every tap before the window, every tap past it, and blends across both track ends."""
    t = np.arange(T)
    return [t - T, 2 * T - 1 - t,
            _tab(np.stack([t - T, 2 * T - 1 - t], 1), np.stack([np.full(T, ONE - 12345), np.full(T, 12345)], 1)),
            _tab(np.stack([t * 0 - 1, t, t + T, t * 0 + 2 * T - 1], 1), np.full((T, 4), ONE // 4))]


def _as_pair(v, T):
    if isinstance(v, tuple):
        return v
    return np.asarray(v, np.int32)[:, None], np.full((T, 1), ONE, np.int32)


def _track(seed, n_frames=200, H=96, W=96, Ta_full=800):
    g = torch.Generator().manual_seed(seed)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8)
    track[::3, : H // 2, : W // 4] = 255                               # saturated patches and hard edges on every third frame
    track[1::3, H // 2:, W // 2:] = 0
    mel = (-80.0 * torch.rand((1, 80, Ta_full), generator=g)).cuda()
    return track.cuda(), mel


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(96, 96), (50, 70)])                  # 50x70: 10 500-byte frames, not 16-byte multiples
@pytest.mark.parametrize("offset", [0, 3])
def test_retime_windows_bytes(model, H, W, offset):
    """The builder's output (lsd_retime_windows) equals the oracle byte for byte: the default ladder, taps clamped below frame 0
    and past the track's end with windows at both ends of the track, random 1- to 4-tap blends; offset 3: a track base that is not
    16-byte aligned (byte loads and stores).  One launch for the whole call."""
    T, n_frames = 32, 45
    g = torch.Generator().manual_seed(H * W + offset)
    host = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8)
    host[::2, : H // 2, : W // 3] = 255
    host[1::2, H // 3:, W // 2:] = 0
    buf = torch.empty(host.numel() + 16, dtype=torch.uint8, device="cuda")
    track = buf[offset:offset + host.numel()].view(n_frames, H, W, 3)
    track.copy_(host)
    starts = [0, 6, n_frames - T]
    variants = P.temporal_variants(T)[1] + _edge_taps(T) + _random_taps(T, 6, seed=H + offset)
    p = lb.Predictor(model, chunk_size=T)
    n0 = model.launch_count()
    out = p.retime_track_windows(track, starts, variants).cpu().numpy()
    assert model.launch_count() == n0 + 1
    assert out.shape == (3, len(variants), T, H, W, 3)
    host = host.numpy()
    for i, s in enumerate(starts):
        for k, v in enumerate(variants):
            assert np.array_equal(out[i, k], rto.retime_window(host, s, *_as_pair(v, T))), (i, k)
    assert np.array_equal(out[:, 0], np.stack([host[s:s + T] for s in starts]))


def _host_reference(p, track, starts, mel, total_v_frames, variants, a_from=None):
    """(n, K) logits: every (window, variant) retimed by the oracle, the windows laid end to end as one track (starts 0, T, 2T, ...)
    and scored by score_track_logits with the window's own audio start."""
    T = p.chunk_size
    host = track.cpu().numpy()
    wins = [rto.retime_window(host, s, *_as_pair(v, T)) for s in starts for v in variants]
    flat = torch.from_numpy(np.concatenate(wins)).cuda()
    a = [s for s in (a_from or starts) for _ in variants]
    ref = p.score_track_logits(flat, [r * T for r in range(len(wins))], mel, total_v_frames, audio_starts_from=a).cpu()
    return ref.view(len(starts), len(variants))


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_retime_bitwise(model, prec):
    """Every (window, variant) logit equals the plain forward of the window retimed by the oracle, with explicit audio starts;
    the `none` column equals score_track_logits.  Windows at both ends of the track read clamped taps."""
    model.compute_precision = prec
    track, mel = _track(91)
    n_frames = 200
    starts = [0, 21, 84, 147, n_frames - 32]
    p = lb.Predictor(model, batch_size=16)
    a_from = [s + 3 for s in starts]
    variants = P.temporal_variants(32)[1] + _edge_taps(32)[2:]
    out = p.score_track_retimes(track, starts, mel, n_frames, variants, audio_starts_from=a_from).cpu()
    assert out.shape == (len(starts), len(variants)) and out.dtype == torch.float32
    assert torch.equal(out, _host_reference(p, track, starts, mel, n_frames, variants, a_from=a_from))
    plain = p.score_track_retimes(track, starts, mel, n_frames, variants)[:, 0].cpu()
    assert torch.equal(plain, p.score_track_logits(track, starts, mel, n_frames).cpu())
    assert not torch.equal(out[:, NAMES_15.index("drift8")], out[:, 0])


def _retimes_raw(model, track, starts, mel, n_frames, variants, batch, ws_bytes, T=32, Ta=128):
    """lsd_score_retimes straight through the C-ABI, in a workspace of exactly ws_bytes, twice on the same workspace."""
    L = _cabi.lib()
    n = len(starts)
    p = lb.Predictor(model)
    K, vc = p._retime_args(track, starts, variants)
    H, W = int(track.shape[1]), int(track.shape[2])
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        L.lsd_workspace_invalidate(h.ptr)
        logits = torch.empty(n, K, dtype=torch.float32, device="cuda")
        for _ in range(2):
            rc = L.lsd_score_retimes(h.ptr, track.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*starts), None, n, T, mel.data_ptr(),
                                     int(mel.shape[1]), int(mel.shape[2]), n_frames, Ta, vc, K, model._precision(), batch,
                                     logits.data_ptr(), ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
            _cabi.check(h.ptr, rc)
            out = logits.cpu()
        L.lsd_workspace_invalidate(h.ptr)
    return out


@pytest.mark.gpu
def test_retime_batches_and_exact_workspace(model):
    """batch=7 over 54 rows (7 full batches and a short one of 5): pipelined in a double workspace and again in exactly the queried
    workspace, both equal to one batch of 64 and to the host reference."""
    model.compute_precision = "bf16"
    track, mel = _track(92)
    n_frames = 200
    starts = list(range(0, 169, 21))                                  # 9 windows
    names, tabs, _ = P.temporal_variants(32)
    variants = [tabs[names.index(k)] for k in ("none", "hold8", "blend10", "freeze10", "drift8", "exposure3")]   # K = 6
    L = _cabi.lib()
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        need7 = L.lsd_score_retimes_workspace_bytes(h.ptr, 7, 6, 32, 96, 96, 80, 128, _cabi.LSD_PREC_BF16)
        need64 = L.lsd_score_retimes_workspace_bytes(h.ptr, 64, 6, 32, 96, 96, 80, 128, _cabi.LSD_PREC_BF16)
    assert 0 < need7 < need64
    one = _retimes_raw(model, track, starts, mel, n_frames, variants, 64, need64)
    piped = _retimes_raw(model, track, starts, mel, n_frames, variants, 7, 2 * need7)
    exact = _retimes_raw(model, track, starts, mel, n_frames, variants, 7, need7)
    assert torch.equal(piped, one) and torch.equal(exact, one)
    p = lb.Predictor(model, batch_size=64)
    assert torch.equal(one, _host_reference(p, track, starts, mel, n_frames, variants))


@pytest.mark.gpu
def test_retime_argument_errors(model):
    """Bad arguments return their status before anything is launched, from both entries."""
    model.compute_precision = "bf16"
    T = 32
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8, device="cuda")
    mel = torch.zeros((1, 80, 300), device="cuda")
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    ws = model._workspace(1 << 20, track.device)
    out = torch.empty(2, 2, device="cuda")
    n0 = model.launch_count()

    def entries(K, mut=None):
        a = np.zeros((max(K, 1), T, 8), np.int32)
        a[:, :, 0] = np.arange(T)
        a[:, :, 4] = ONE
        if mut:
            mut(a)
        return (_cabi.LsdRetime * (max(K, 1) * T)).from_buffer_copy(a.tobytes())

    def call(vc, K, starts=(0, 8), n=2, null_track=False):
        trk = None if null_track else track.data_ptr()
        st = (C.c_int32 * max(n, 1))(*starts[:max(n, 1)])
        rc = L.lsd_score_retimes(h.ptr, trk, 64, 96, 96, st, None, n, T, mel.data_ptr(), 80, 300,
                                 64, 128, vc, K, _cabi.LSD_PREC_BF16, 2, out.data_ptr(), ws.data_ptr(), ws.numel(), None)
        wrc = L.lsd_retime_windows(h.ptr, trk, 64, 96, 96, st, n, T, vc, K, out.data_ptr(), ws.data_ptr(), ws.numel(), None)
        assert wrc == rc, (rc, wrc)
        return rc

    def set_(idx, val):
        def f(a):
            a[idx] = val
        return f

    ok = entries(1)
    assert call(None, 1) == _cabi.LSD_ERR_ARG
    assert call(ok, 1, null_track=True) == _cabi.LSD_ERR_ARG
    assert call(ok, 0) == _cabi.LSD_ERR_SHAPE
    assert call(entries(65), 65) == _cabi.LSD_ERR_SHAPE
    assert call(ok, 1, starts=(0, 33)) == _cabi.LSD_ERR_SHAPE                            # window [33, 65) outside the 64-frame track
    assert call(ok, 1, starts=(-1, 0)) == _cabi.LSD_ERR_SHAPE
    assert call(entries(1, set_((0, 3, 0), -T - 1)), 1) == _cabi.LSD_ERR_SHAPE           # src below -T
    assert call(entries(1, set_((0, 3, 0), 2 * T)), 1) == _cabi.LSD_ERR_SHAPE            # src past 2T - 1
    assert call(entries(1, set_((0, 5, 2), 2 * T)), 1) == _cabi.LSD_ERR_SHAPE            # ... on a tap of weight 0
    assert call(entries(2, set_((1, 7, slice(4, 6)), [ONE + 1, -1])), 2) == _cabi.LSD_ERR_ARG   # a negative weight
    assert call(entries(2, set_((1, 31, 4), ONE - 1)), 2) == _cabi.LSD_ERR_ARG           # weights sum to 32767
    assert call(entries(1, set_((0, 0, slice(4, 8)), [ONE, ONE, 0, 0])), 1) == _cabi.LSD_ERR_ARG
    assert call(entries(64), 64, n=(2 ** 31 - 1) // (64 * T) + 1) == _cabi.LSD_ERR_SHAPE   # n * K * T above INT32_MAX
    assert model.launch_count() == n0
    assert call(ok, 1, n=0) == _cabi.LSD_OK and model.launch_count() == n0


@pytest.mark.gpu
def test_temporal_track_matches_its_logits(model):
    model.compute_precision = "bf16"
    track, mel = _track(93)
    n_frames = 200
    starts = list(range(0, 169, 24))                                   # 8 windows
    p = lb.Predictor(model, batch_size=64)
    rt = p.temporal_track(track, starts, mel, n_frames, confidence_threshold=0.5)
    names, tabs, rates = P.temporal_variants(32)
    assert rt["variants"] == names and rt["rates"] == rates and rt["window_starts"] == starts
    logits = p.score_track_retimes(track, starts, mel, n_frames, tabs).cpu().numpy()
    probs = np.array([[p._calibrate(float(x)) for x in row] for row in logits])
    want = augmentation_stability(probs, 0.5, p.confidence_smoothing, p.trim_ratio)
    for k, v in want.items():
        assert np.array_equal(np.asarray(rt[k]), np.asarray(v)), k
    assert rt["lowest_stable_fps"] == lowest_stable_quality(rates, want["variant_confidence"], want["confidence"], 0.5)
    plain = [p._calibrate(float(x)) for x in p.score_track_logits(track, starts, mel, n_frames).cpu().tolist()]
    assert rt["confidence"] == p._robust_confidence(plain)


@pytest.mark.gpu
def test_long_video_temporal_entry_on_gpu(model):
    """temporal=True: `confidence` is the selected track's plain window aggregate, every other result key is unchanged."""
    model.compute_precision = "bf16"
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(model, batch_size=16)
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, temporal=True)
    assert set(res) == set(base) | {"temporal"}
    tp = res["temporal"]
    sel = next(t for t in res["tracks"] if t["track_id"] == res["selected_track_id"])
    assert tp["track_id"] == res["selected_track_id"]
    assert tp["confidence"] == pred._robust_confidence(sel["window_confidences"])
    tr = next(t for t in tracks if int(t["track_id"]) == tp["track_id"])
    assert tp["window_starts"] == [int(s) for s in tr["chunk_starts"]]
    names, _, rates = P.temporal_variants(32, spec["fps"])
    assert tp["variants"] == names and tp["rates"] == rates and len(tp["variant_confidence"]) == len(names)
    for k in base:
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k


@pytest.mark.gpu
def test_long_video_temporal_chunks_match_crops(model):
    """The default temporal hook on the reference's chunk format gives the same report, bit for bit, as on the same frames given as
    `crops_u8`: frames outside a window are the video's own frames, not the overlapping next window's."""
    model.compute_precision = "bf16"
    spec = SCENARIOS["two_tracks_clear_winner"]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(model, batch_size=64)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, temporal=True)
    chunked = [_as_chunks(t) for t in tracks]
    res_ch = lb.predict_long_video_from_tracks(pred, chunked, mel, vad, spec["fps"], n_frames, temporal=True)
    assert res_ch["selected_track_id"] == res["selected_track_id"]
    assert json.dumps(res_ch["temporal"], sort_keys=True, default=str) == json.dumps(res["temporal"], sort_keys=True, default=str)
