"""Resolution robustness: `Predictor.score_track_resizes` (lsd_score_resizes), `Predictor.resize_track_windows` (lsd_resize_windows),
`Predictor.resolution_track` and the `resolution` entry of `predict_long_video_from_tracks`.  Every frame of a variant is
cv2.resize(cv2.resize(frame, (w, h), INTER_AREA), (W, H), INTER_LINEAR): oracle/resize_oracle.py restates it and is checked against
cv2 here; the logit of (window, variant) must be bit for bit the plain forward's logit for that window resized on the host by the
oracle."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import augmentation_stability, lowest_stable_quality
from oracle import resize_oracle as ro
from tests.golden.long_video_synth import SCENARIOS, make_audio, make_tracks

P = lb.Predictor
LADDER = [(80, 80), (64, 64), (56, 56), (48, 48), (40, 40), (32, 32), (24, 24)]
# the plain copy, the default ladder, the extremes and mixed integer / non-integer axes
SIZES_96 = [(96, 96)] + LADDER + [(1, 1), (95, 95), (40, 72), (48, 37), (96, 50), (31, 96), (1, 96)]


def _cv2_down_up(cv2, frame, h, w):
    H, W = frame.shape[:2]
    return cv2.resize(cv2.resize(frame, (w, h), interpolation=cv2.INTER_AREA), (W, H), interpolation=cv2.INTER_LINEAR)


def _smooth(rng, H, W):
    import cv2
    return cv2.resize(rng.integers(0, 256, (max(1, H // 8), max(1, W // 8), 3), dtype=np.uint8), (W, H), interpolation=cv2.INTER_CUBIC)


def _hard(rng, H, W):
    """Saturated 0 / 255 patches, hard colour edges and a one-pixel checkerboard: the rounding and saturation of both passes."""
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    img[: H // 2, : W // 3] = (255, 0, 0)
    img[H // 2:, : W // 3] = (0, 0, 255)
    img[:, W // 3: W // 2] = 255
    img[H // 4: 3 * H // 4, W // 2: 3 * W // 4] = 0
    img[::2, 3 * W // 4:] = (0, 255, 255)
    img[1::2, 3 * W // 4:] = (255, 0, 255)
    img[::2, 3 * W // 4::2] = 0
    return img


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("h", range(1, 97))
def test_oracle_matches_cv2_every_size(h):
    """Every face size h x w, 1 <= h, w <= 96, of a 96x96 frame (square and non-square: every mix of ratio-2, integer and
    non-integer axes), on random content; the down pass alone too."""
    cv2 = pytest.importorskip("cv2")
    img = np.random.default_rng(h).integers(0, 256, (96, 96, 3), dtype=np.uint8)
    for w in range(1, 97):
        assert np.array_equal(ro.downscale_area(img, h, w), cv2.resize(img, (w, h), interpolation=cv2.INTER_AREA)), (h, w)
        assert np.array_equal(ro.down_up(img, h, w), _cv2_down_up(cv2, img, h, w)), (h, w)


@pytest.mark.parametrize("H,W", [(96, 96), (64, 80), (112, 96)])
def test_oracle_matches_cv2_shapes_and_content(H, W):
    """Random, smooth and saturated / hard-edged crops, every square face size and a spread of non-square ones."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(H * W)
    sizes = [(s, s) for s in range(1, min(H, W) + 1)] + [(h, w) for h in range(1, H + 1, 5) for w in range(1, W + 1, 7)]
    sizes += [(H, w) for w in range(1, W + 1, 3)] + [(h, W) for h in range(1, H + 1, 3)]
    for img in (_smooth(rng, H, W), _hard(rng, H, W)):
        for h, w in sizes:
            assert np.array_equal(ro.down_up(img, h, w), _cv2_down_up(cv2, img, h, w)), (H, W, h, w)


def test_oracle_paths_and_plain_copy():
    """The default ladder of a 96x96 crop takes all three INTER_AREA paths; the crop size is the frame itself."""
    assert ro.area_integer_ratio(96, 48) == 2
    assert ro.area_integer_ratio(96, 32) == 3 and ro.area_integer_ratio(96, 24) == 4
    assert [ro.area_integer_ratio(96, s) for s in (80, 64, 56, 40)] == [0, 0, 0, 0]
    img = _hard(np.random.default_rng(3), 96, 96)
    assert np.array_equal(ro.down_up(img, 96, 96), img)
    # ratio 2 rounds half up ((sum + 2) >> 2), other integer ratios half to even: a 2x2 block summing to 2 gives 1
    blk = np.zeros((2, 2, 3), np.uint8)
    blk[0, 0] = 2
    assert ro.downscale_area(blk, 1, 1)[0, 0, 0] == 1


def _tables(variants, H, W):
    L = _cabi.lib()
    vc = (_cabi.LsdResize * len(variants))(*[_cabi.LsdResize(h, w) for h, w in variants])
    n = L.lsd_resize_tables(vc, len(variants), H, W, None)
    assert n == len(variants) * (10 + 9 * (H + W))
    out = np.zeros(n, np.int32)
    assert L.lsd_resize_tables(vc, len(variants), H, W, out.ctypes.data) == n
    return out.reshape(len(variants), -1)


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()


@pytest.mark.parametrize("H,W", [(96, 96), (64, 80), (50, 70)])
def test_host_tables_equal_oracle(built, H, W):
    """lsd_resize_tables (what the kernel reads) against the oracle's taps, field by field."""
    sizes = [(H, W)] + P.resolution_variants(H, W)[1][1:] + [(1, 1), (H - 1, W - 1), (H, 1), (1, W), (H // 2, W // 3), (H - 7, W // 2)]
    tabs = _tables(sizes, H, W)
    as_f32 = lambda a: np.asarray(a, np.int32).view(np.float32)
    for (h, w), t in zip(sizes, tabs):
        xs, xi, xw = 8, 8 + W + 1, 8 + 3 * W + 1
        ys, yi, yw = 8 + 5 * W + 1, 8 + 5 * W + H + 2, 8 + 5 * W + 3 * H + 2
        lx, ly = 8 + 5 * W + 5 * H + 2, 8 + 9 * W + 5 * H + 2
        assert (t[1], t[2]) == (h, w)
        if (h, w) == (H, W):
            assert t[0] == 0
            continue
        kx, ky = ro.area_integer_ratio(W, w), ro.area_integer_ratio(H, h)
        if kx and ky:
            assert t[0] == (1 if kx == ky == 2 else 2) and (t[3], t[4]) == (kx, ky)
            assert as_f32([t[5]])[0] == np.float32(1.0) / np.float32(kx * ky)
        else:
            assert t[0] == 3
            for start, si, wt, src, dst in ((xs, xi, xw, W, w), (ys, yi, yw, H, h)):
                taps = ro.area_taps(src, dst)
                n = len(taps)
                assert n <= 2 * src
                assert t[start + dst] == n
                assert [int(v) for v in t[start:start + dst + 1]] == [sum(1 for d, _, _ in taps if d < e) for e in range(dst + 1)]
                assert [int(v) for v in t[si:si + n]] == [s for _, s, _ in taps]
                assert np.array_equal(as_f32(t[wt:wt + n]), np.array([x for _, _, x in taps], np.float32))
        for base, src, dst, clamp in ((lx, w, W, True), (ly, h, H, False)):
            want = ro.linear_taps(src, dst, clamp)
            for j in range(4):
                assert np.array_equal(t[base + j * dst: base + (j + 1) * dst], want[j]), (h, w, base, j)


def test_host_table_errors(built):
    L = _cabi.lib()
    ok = (_cabi.LsdResize * 1)(_cabi.LsdResize(48, 48))
    assert L.lsd_resize_tables(None, 1, 96, 96, None) == _cabi.LSD_ERR_ARG
    assert L.lsd_resize_tables(ok, 0, 96, 96, None) == _cabi.LSD_ERR_SHAPE
    assert L.lsd_resize_tables((_cabi.LsdResize * 1)(_cabi.LsdResize(97, 48)), 1, 96, 96, None) == _cabi.LSD_ERR_SHAPE
    assert L.lsd_resize_tables((_cabi.LsdResize * 1)(_cabi.LsdResize(48, 0)), 1, 96, 96, None) == _cabi.LSD_ERR_SHAPE
    assert L.lsd_resize_tables(ok, 1, 256, 256, None) == _cabi.LSD_ERR_SHAPE          # beyond 227 KB of shared memory


def test_default_resolution_variants():
    names, sizes = P.resolution_variants(96, 96)
    assert names == ["none", "80x80", "64x64", "56x56", "48x48", "40x40", "32x32", "24x24"]
    assert sizes == [(96, 96)] + LADDER
    names, sizes = P.resolution_variants(64, 80)
    assert sizes == [(64, 80), (53, 67), (43, 53), (37, 47), (32, 40), (27, 33), (21, 27), (16, 20)] and len(names) == 8


def test_lowest_stable_side_hand_built(monkeypatch):
    """resolution_track's report from hand-built logits (the same logit in every window of a column)."""
    pred = P(None, device=torch.device("cpu"))
    track = torch.zeros((40, 96, 96, 3), dtype=torch.uint8)
    mel = torch.zeros((1, 80, 200))

    def run(cols):
        monkeypatch.setattr(pred, "score_track_resizes", lambda *a, **k: torch.tensor([cols] * 3, dtype=torch.float32))
        return pred.resolution_track(track, [0, 4, 8], mel, 40, confidence_threshold=0.5)

    res = run([4.0, 4.0, 3.0, 2.0, 1.0, 0.5, 0.2, 0.1])
    assert res["lowest_stable_side"] == 24 and res["verdict_stable"]
    assert res["sizes"] == [(96, 96)] + LADDER and res["variants"][0] == "none" and res["window_starts"] == [0, 4, 8]
    assert run([4.0, 4.0, 3.0, 2.0, -1.0, 0.5, -0.2, -0.1])["lowest_stable_side"] == 56          # flips at 48
    assert run([4.0, -4.0, 3.0, 2.0, 1.0, 0.5, 0.2, 0.1])["lowest_stable_side"] is None          # the largest face flips
    res = run([-3.0, -3.0, -2.0, -1.0, -0.5, -0.1, 0.3, 0.2])                                 # a fake verdict
    assert res["lowest_stable_side"] == 40 and not res["verdict_stable"]
    probs = np.array([[pred._calibrate(x) for x in [-3.0, -3.0, -2.0, -1.0, -0.5, -0.1, 0.3, 0.2]]] * 3)
    want = augmentation_stability(probs, 0.5, pred.confidence_smoothing, pred.trim_ratio)
    for k, v in want.items():
        assert np.array_equal(np.asarray(res[k]), np.asarray(v)), k
    assert res["lowest_stable_side"] == lowest_stable_quality([None, 80, 64, 56, 48, 40, 32, 24], want["variant_confidence"],
                                                              want["confidence"], 0.5)


@pytest.mark.parametrize("variants", [[], [(48, 48)] * 65, [(0, 48)], [(48, 0)], [(97, 48)], [(48, 97)], [(48.0, 48)], [(48,)],
                                      [(48, 48, 3)]])
def test_argument_errors_raise_value_error(variants):
    pred = P(None, device=torch.device("cpu"))
    track = torch.zeros((40, 96, 96, 3), dtype=torch.uint8)
    mel = torch.zeros((1, 80, 200))
    with pytest.raises(ValueError):
        pred.score_track_resizes(track, [0], mel, 40, variants)
    with pytest.raises(ValueError):
        pred.resize_track_windows(track, [0], variants)


def test_argument_errors_track_window_and_audio():
    pred = P(None, device=torch.device("cpu"))
    track = torch.zeros((40, 96, 96, 3), dtype=torch.uint8)
    mel = torch.zeros((1, 80, 200))
    with pytest.raises(ValueError):
        pred.resize_track_windows(track, [9], [(48, 48)])                  # window [9, 41) outside the 40-frame track
    with pytest.raises(ValueError):
        pred.resize_track_windows(track.float(), [0], [(48, 48)])
    with pytest.raises(ValueError):
        pred.resize_track_windows(track[..., :2], [0], [(48, 48)])
    with pytest.raises(ValueError):
        pred.score_track_resizes(track, [0], mel[0], 40, [(48, 48)])
    with pytest.raises(ValueError):
        pred.score_track_resizes(track, [0, 4], mel, 40, [(48, 48)], audio_starts_from=[0])
    assert pred._resize_args(track, [0, 8], [(96, 96), (1, 1), (np.int64(40), 72)])[0] == 3


def test_long_video_resolution_entry():
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def resolution_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"confidence": 0.7, "lowest_stable_side": 40, "window_starts": [int(s) for s in tr["chunk_starts"]]}

    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, resolution=True,
                                            resolution_fn=resolution_fn, **fns)
    assert "resolution" not in base
    assert set(res) == set(base) | {"resolution"}
    assert res["resolution"]["track_id"] == res["selected_track_id"] == seen[0] and len(seen) == 1
    assert res["resolution"]["lowest_stable_side"] == 40
    tr = next(t for t in tracks if int(t["track_id"]) == seen[0])
    assert res["resolution"]["window_starts"] == [int(s) for s in tr["chunk_starts"]]
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def model(built, seed0_sd):
    m = lb.LipSyncModel()
    m.load_state_dict(seed0_sd, strict=True)
    return m.to("cuda:0").eval()


def _track(seed, n_frames=200, H=96, W=96, Ta_full=800):
    g = torch.Generator().manual_seed(seed)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8)
    track[::3, : H // 2, : W // 4] = 255                               # saturated patches and hard edges on every third frame
    track[1::3, H // 2:, W // 2:] = 0
    mel = (-80.0 * torch.rand((1, 80, Ta_full), generator=g)).cuda()
    return track.cuda(), mel


def _score_windows_explicit(p, track, starts, mel, total_v_frames, a_starts, chunk_a_size):
    """lsd_score_windows with explicit audio starts (the first mel column of every window, used as given)."""
    m = p.model
    n = len(starts)
    out = torch.empty(n, dtype=torch.float32, device="cuda")
    with m._lsd_lock:
        h = m._ensure_handle(m._device())
        L = _cabi.lib()
        prec = m._precision()
        batch = min(p.batch_size, n)
        need = L.lsd_score_workspace_bytes(h.ptr, batch, p.chunk_size, track.shape[1], track.shape[2], mel.shape[1], chunk_a_size, prec)
        ws = m._workspace(2 * need, m._device())
        rc = L.lsd_score_windows(h.ptr, track.data_ptr(), int(track.shape[0]), int(track.shape[1]), int(track.shape[2]),
                                 (C.c_int32 * n)(*starts), (C.c_int32 * n)(*[int(x) for x in a_starts]), n, p.chunk_size, mel.data_ptr(),
                                 int(mel.shape[1]), int(mel.shape[2]), total_v_frames, chunk_a_size, prec, batch, out.data_ptr(), ws.data_ptr(),
                                 ws.numel(), torch.cuda.current_stream().cuda_stream)
        _cabi.check(h.ptr, rc)
    return out.cpu()


def _host_reference(p, track, starts, mel, total_v_frames, variants, a_from=None, chunk_a_size=128):
    """(n, K) logits: every (window, variant) resized by the oracle, the windows laid end to end as one track and scored by
    lsd_score_windows with the window's own audio start."""
    T = p.chunk_size
    host = track.cpu().numpy()
    wins = [ro.down_up_window(host[s:s + T], h, w) for s in starts for h, w in variants]
    flat = torch.from_numpy(np.concatenate(wins)).cuda()
    a = [p._audio_start(s, int(mel.shape[2]), total_v_frames, chunk_a_size) for s in (a_from or starts) for _ in variants]
    ref = _score_windows_explicit(p, flat, [r * T for r in range(len(wins))], mel, total_v_frames, a, chunk_a_size)
    return ref.view(len(starts), len(variants))


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,sizes", [
    (96, 96, SIZES_96),
    (64, 80, [(64, 80), (53, 67), (43, 53), (32, 40), (16, 20), (32, 80), (64, 40), (1, 1), (63, 79), (40, 72), (48, 37)]),
    (50, 70, [(50, 70), (25, 35), (10, 14), (40, 56), (1, 1), (49, 69), (17, 70)]),     # 10 500-byte frames: not 16-byte multiples
])
@pytest.mark.parametrize("offset", [0, 3])
def test_resize_windows_bytes(model, H, W, sizes, offset):
    """The builder's output (lsd_resize_windows) equals the oracle byte for byte: the default ladder, 1x1, one pixel short of the
    crop, non-square sizes, the plain copy; offset 3: a track base that is not 16-byte aligned (byte loads and stores)."""
    T, n_frames = 4, 11
    g = torch.Generator().manual_seed(H * W + offset)
    host = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8)
    host[::2, : H // 2, : W // 3] = 255
    host[1::2, H // 3:, W // 2:] = 0
    buf = torch.empty(host.numel() + 16, dtype=torch.uint8, device="cuda")
    track = buf[offset:offset + host.numel()].view(n_frames, H, W, 3)
    track.copy_(host)
    starts = [0, 3, 7]
    p = lb.Predictor(model, chunk_size=T)
    n0 = model.launch_count()
    out = p.resize_track_windows(track, starts, sizes).cpu().numpy()
    assert model.launch_count() == n0 + 1
    host = host.numpy()
    for i, s in enumerate(starts):
        for k, (h, w) in enumerate(sizes):
            assert np.array_equal(out[i, k], ro.down_up_window(host[s:s + T], h, w)), (i, k, h, w)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_resize_bitwise(model, prec):
    """Every (window, variant) logit equals the plain forward of the window resized by the oracle, with explicit audio starts;
    the plain column equals score_track_logits."""
    model.compute_precision = prec
    track, mel = _track(81)
    n_frames = 200
    starts = list(range(0, n_frames - 32 + 1, 21))                   # 9 windows x 8 variants: 72 rows, 5 batches of 16
    p = lb.Predictor(model, batch_size=16)
    a_from = [s + 3 for s in starts]
    _, sizes = P.resolution_variants(96, 96)
    out = p.score_track_resizes(track, starts, mel, n_frames, sizes, audio_starts_from=a_from).cpu()
    assert out.shape == (len(starts), len(sizes)) and out.dtype == torch.float32
    assert torch.equal(out, _host_reference(p, track, starts, mel, n_frames, sizes, a_from=a_from))
    plain = p.score_track_resizes(track, starts, mel, n_frames, sizes)[:, 0].cpu()
    assert torch.equal(plain, p.score_track_logits(track, starts, mel, n_frames).cpu())
    assert not torch.equal(out[:, 7], out[:, 0])


def _resizes_raw(model, track, starts, mel, n_frames, variants, batch, ws_bytes, T=32, Ta=128):
    """lsd_score_resizes straight through the C-ABI, in a workspace of exactly ws_bytes, twice on the same workspace."""
    L = _cabi.lib()
    n, K = len(starts), len(variants)
    H, W = int(track.shape[1]), int(track.shape[2])
    vc = (_cabi.LsdResize * K)(*[_cabi.LsdResize(h, w) for h, w in variants])
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        L.lsd_workspace_invalidate(h.ptr)
        logits = torch.empty(n, K, dtype=torch.float32, device="cuda")
        for _ in range(2):
            rc = L.lsd_score_resizes(h.ptr, track.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*starts), None, n, T, mel.data_ptr(),
                                     int(mel.shape[1]), int(mel.shape[2]), n_frames, Ta, vc, K, model._precision(), batch,
                                     logits.data_ptr(), ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
            _cabi.check(h.ptr, rc)
            out = logits.cpu()
        L.lsd_workspace_invalidate(h.ptr)
    return out


@pytest.mark.gpu
def test_resize_batches_and_exact_workspace(model):
    """batch=7 over 54 rows (7 full batches and a short one of 5): pipelined in a double workspace and again in exactly the queried
    workspace, both equal to one batch of 64 and to the host reference."""
    model.compute_precision = "bf16"
    track, mel = _track(82)
    n_frames = 200
    starts = list(range(0, 169, 21))                                  # 9 windows
    variants = [(80, 80), (48, 48), (40, 72), (24, 24), (1, 1), (96, 96)]     # K = 6
    L = _cabi.lib()
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        need7 = L.lsd_score_resizes_workspace_bytes(h.ptr, 7, 6, 32, 96, 96, 80, 128, _cabi.LSD_PREC_BF16)
        need64 = L.lsd_score_resizes_workspace_bytes(h.ptr, 64, 6, 32, 96, 96, 80, 128, _cabi.LSD_PREC_BF16)
    assert 0 < need7 < need64
    one = _resizes_raw(model, track, starts, mel, n_frames, variants, 64, need64)
    piped = _resizes_raw(model, track, starts, mel, n_frames, variants, 7, 2 * need7)
    exact = _resizes_raw(model, track, starts, mel, n_frames, variants, 7, need7)
    assert torch.equal(piped, one) and torch.equal(exact, one)
    p = lb.Predictor(model, batch_size=64)
    assert torch.equal(one, _host_reference(p, track, starts, mel, n_frames, variants))


@pytest.mark.gpu
def test_resize_argument_errors(model):
    """Bad arguments return their status before anything is launched."""
    model.compute_precision = "bf16"
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8, device="cuda")
    mel = torch.zeros((1, 80, 300), device="cuda")
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    ws = model._workspace(1 << 20, track.device)
    out = torch.empty(2, 2, device="cuda")
    n0 = model.launch_count()

    def call(variants, K=None, starts=(0, 8), HW=(96, 96), null=False, null_track=False):
        K = len(variants) if K is None else K
        vc = None if null else (_cabi.LsdResize * max(K, 1))(*[_cabi.LsdResize(a, b) for a, b in variants][:max(K, 1)])
        trk = None if null_track else track.data_ptr()
        rc = L.lsd_score_resizes(h.ptr, trk, 64, HW[0], HW[1], (C.c_int32 * 2)(*starts), None, 2, 32, mel.data_ptr(), 80, 300,
                                 64, 128, vc, K, _cabi.LSD_PREC_BF16, 2, out.data_ptr(), ws.data_ptr(), ws.numel(), None)
        wrc = L.lsd_resize_windows(h.ptr, trk, 64, HW[0], HW[1], (C.c_int32 * 2)(*starts), 2, 32, vc, K, out.data_ptr(),
                                   ws.data_ptr(), ws.numel(), None)
        assert wrc == rc
        return rc

    ok = (48, 48)
    assert call([ok], null=True) == _cabi.LSD_ERR_ARG
    assert call([ok], null_track=True) == _cabi.LSD_ERR_ARG
    assert call([ok], K=0) == _cabi.LSD_ERR_SHAPE
    assert call([ok] * 65) == _cabi.LSD_ERR_SHAPE
    assert call([ok, (0, 48)]) == _cabi.LSD_ERR_SHAPE
    assert call([ok, (48, 0)]) == _cabi.LSD_ERR_SHAPE
    assert call([(97, 48)]) == _cabi.LSD_ERR_SHAPE
    assert call([(48, 97)]) == _cabi.LSD_ERR_SHAPE
    assert call([(96, 96)], HW=(96, 80)) == _cabi.LSD_ERR_SHAPE            # a face size wider than the crop
    assert call([ok], HW=(256, 256)) == _cabi.LSD_ERR_SHAPE                # beyond 227 KB of shared memory
    assert call([ok], starts=(0, 33)) == _cabi.LSD_ERR_SHAPE               # window [33, 65) outside the 64-frame track
    assert call([(96, 96)], starts=(0, 33)) == _cabi.LSD_ERR_SHAPE
    assert model.launch_count() == n0


@pytest.mark.gpu
def test_resolution_track_matches_its_logits(model):
    model.compute_precision = "bf16"
    track, mel = _track(83)
    n_frames = 200
    starts = list(range(0, 169, 24))                                   # 8 windows
    p = lb.Predictor(model, batch_size=64)
    rt = p.resolution_track(track, starts, mel, n_frames, confidence_threshold=0.5)
    names, sizes = P.resolution_variants(96, 96)
    assert rt["variants"] == names and rt["sizes"] == sizes and rt["window_starts"] == starts
    logits = p.score_track_resizes(track, starts, mel, n_frames, sizes).cpu().numpy()
    probs = np.array([[p._calibrate(float(x)) for x in row] for row in logits])
    want = augmentation_stability(probs, 0.5, p.confidence_smoothing, p.trim_ratio)
    for k, v in want.items():
        assert np.array_equal(np.asarray(rt[k]), np.asarray(v)), k
    heights = [None] + [h for h, _ in sizes[1:]]
    assert rt["lowest_stable_side"] == lowest_stable_quality(heights, want["variant_confidence"], want["confidence"], 0.5)
    plain = [p._calibrate(float(x)) for x in p.score_track_logits(track, starts, mel, n_frames).cpu().tolist()]
    assert rt["confidence"] == p._robust_confidence(plain)


@pytest.mark.gpu
def test_long_video_resolution_entry_on_gpu(model):
    """resolution=True: `confidence` is the selected track's plain window aggregate, every other result key is unchanged."""
    model.compute_precision = "bf16"
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(model, batch_size=16)
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, resolution=True)
    assert set(res) == set(base) | {"resolution"}
    rs = res["resolution"]
    sel = next(t for t in res["tracks"] if t["track_id"] == res["selected_track_id"])
    assert rs["track_id"] == res["selected_track_id"]
    assert rs["confidence"] == pred._robust_confidence(sel["window_confidences"])
    tr = next(t for t in tracks if int(t["track_id"]) == rs["track_id"])
    assert rs["window_starts"] == [int(s) for s in tr["chunk_starts"]]
    assert len(rs["variant_confidence"]) == 8
    for k in base:
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k
