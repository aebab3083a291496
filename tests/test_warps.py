"""Crop-jitter robustness: `Predictor.score_track_warps` (lsd_score_warps), the matrix helpers, `Predictor.robustness_track`,
`aggregate.augmentation_stability` and the `robustness` entry of `predict_long_video_from_tracks`.
The re-crop is cv2.warpAffine(INTER_LINEAR, BORDER_REPLICATE): oracle/warp_oracle.py restates it and is checked against cv2 here;
the logit of (window, variant) must be bit for bit the plain forward's logit for that window warped on the host by the oracle."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import augmentation_stability
from oracle import warp_oracle as wo
from tests.golden.long_video_synth import SCENARIOS, make_audio, make_tracks

P = lb.Predictor


def _variants(T, H, W):
    """(K, T, 2, 3): identity, flip, sub-pixel shift, shifts and a zoom-out that push taps past every border, rotation + scale,
    and a per-frame jitter."""
    ssr = P.shift_scale_rotate_warp
    fixed = [ssr(H, W), P.flip_warp(W), ssr(H, W, dx=0.40625, dy=-0.71875), ssr(H, W, dx=-30, dy=25), ssr(H, W, dx=21.5, dy=-27.25),
             ssr(H, W, scale=0.8, angle_deg=15), ssr(H, W, dx=2, scale=1.25, angle_deg=-9)]
    mats = [np.broadcast_to(M, (T, 2, 3)) for M in fixed] + [P.jitter_warps(T, H, W, 1.5, 0.02, 7)]
    return np.stack(mats)


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()


@pytest.fixture(scope="module")
def model(built, seed0_sd):
    m = lb.LipSyncModel()
    m.load_state_dict(seed0_sd, strict=True)
    return m.to("cuda:0").eval()


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


def _host_reference(p, track, starts, mel, total_v_frames, mats, chunk_a_size=128):
    """(n, K) logits: every (window, variant) warped by the oracle, the warped windows laid end to end as one track and scored by
    lsd_score_windows with the window's own audio start."""
    T = p.chunk_size
    host = track.cpu().numpy()
    wins = [wo.warp_window(host[s:s + T], M) for s in starts for M in mats]
    flat = torch.from_numpy(np.concatenate(wins)).cuda()
    a = [p._audio_start(s, int(mel.shape[2]), total_v_frames, chunk_a_size) for s in starts for _ in mats]
    ref = _score_windows_explicit(p, flat, [r * T for r in range(len(wins))], mel, total_v_frames, a, chunk_a_size)
    return ref.view(len(starts), len(mats))


def _track(seed, n_frames=200, H=96, W=96, Ta_full=800):
    g = torch.Generator().manual_seed(seed)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    mel = (-80.0 * torch.rand((1, 80, Ta_full), generator=g)).cuda()
    return track, mel


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_warps_bitwise(model, prec):
    """Every (window, variant) logit equals the plain forward of the window warped by the oracle; the identity column equals
    score_track_logits and the flip column differs from it."""
    model.compute_precision = prec
    track, mel = _track(61)
    n_frames = 200
    starts = list(range(0, n_frames - 32 + 1, 21))                   # 9 windows x 8 variants: 72 rows, 5 batches of 16 (pipelined on bf16)
    p = lb.Predictor(model, batch_size=16)
    mats = _variants(32, 96, 96)
    out = p.score_track_warps(track, starts, mel, n_frames, mats).cpu()
    assert out.shape == (len(starts), len(mats)) and out.dtype == torch.float32
    ref = _host_reference(p, track, starts, mel, n_frames, mats)
    for k in range(len(mats)):
        assert torch.equal(out[:, k], ref[:, k]), (k, out[:, k], ref[:, k])
    assert torch.equal(out[:, 0], p.score_track_logits(track, starts, mel, n_frames).cpu())
    assert not torch.equal(out[:, 1], out[:, 0])
    # (K, 2, 3) is the same matrix on every frame
    two = p.score_track_warps(track, starts[:3], mel, n_frames, mats[:4, 0]).cpu()
    assert torch.equal(two, out[:3, :4])


def _warps_raw(model, track, starts, mel, n_frames, mats, batch, ws_bytes, T=32, Ta=128):
    """lsd_score_warps straight through the C-ABI, in a workspace of exactly ws_bytes.  Called twice on the same workspace: the
    second call must give the same logits in a workspace an earlier call has already written."""
    L = _cabi.lib()
    n, K = len(starts), len(mats)
    H, W = int(track.shape[1]), int(track.shape[2])
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        L.lsd_workspace_invalidate(h.ptr)
        logits = torch.empty(n, K, dtype=torch.float32, device="cuda")
        wc = (_cabi.LsdWarp * (K * T)).from_buffer_copy(np.ascontiguousarray(mats, dtype=np.float64).tobytes())
        for _ in range(2):
            rc = L.lsd_score_warps(h.ptr, track.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*starts), None, n, T, mel.data_ptr(),
                                   int(mel.shape[1]), int(mel.shape[2]), n_frames, Ta, wc, K, model._precision(), batch, logits.data_ptr(),
                                   ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
            _cabi.check(h.ptr, rc)
            out = logits.cpu()
        L.lsd_workspace_invalidate(h.ptr)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["aligned", "misaligned", "l2_taps"])
def test_warps_batches_and_exact_workspace(model, route, monkeypatch):
    """batch=7 over 54 rows (7 full batches and a short one of 5): pipelined in a double workspace and again in exactly the queried
    workspace, both equal to one batch of 64.  misaligned: a track that is not 16-byte aligned stages its frames byte by byte
    instead of with one bulk copy.  l2_taps: LSD_WARP_L2_TAPS makes the kernel read its taps from global memory, the route of
    frames too large for shared memory."""
    model.compute_precision = "bf16"
    n_frames, H, W = 200, 96, 96
    g = torch.Generator().manual_seed(62)
    data = torch.randint(0, 256, (n_frames * H * W * 3 + 16,), generator=g, dtype=torch.uint8).cuda()
    o = 3 if route == "misaligned" else 0
    track = data[o:o + n_frames * H * W * 3].view(n_frames, H, W, 3)
    mel = (-80.0 * torch.rand((1, 80, 800), generator=g)).cuda()
    starts = list(range(0, 169, 21))                                  # 9 windows
    mats = _variants(32, H, W)[1:7]                                   # K = 6
    if route == "l2_taps":
        monkeypatch.setenv("LSD_WARP_L2_TAPS", "1")
    L = _cabi.lib()
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        need7 = L.lsd_score_warps_workspace_bytes(h.ptr, 7, 6, 32, H, W, 80, 128, _cabi.LSD_PREC_BF16)
        need64 = L.lsd_score_warps_workspace_bytes(h.ptr, 64, 6, 32, H, W, 80, 128, _cabi.LSD_PREC_BF16)
    assert 0 < need7 < need64
    one = _warps_raw(model, track, starts, mel, n_frames, mats, 64, need64)
    piped = _warps_raw(model, track, starts, mel, n_frames, mats, 7, 2 * need7)
    exact = _warps_raw(model, track, starts, mel, n_frames, mats, 7, need7)
    assert torch.equal(piped, one) and torch.equal(exact, one)
    p = lb.Predictor(model, batch_size=64)
    assert torch.equal(one, _host_reference(p, track.contiguous(), starts, mel, n_frames, mats))


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,offset,l2", [
    (40, 56, 0, False),     # W % 16 != 0: a thread's 16 pixels wrap across rows; bulk staging, 16-byte stores
    (37, 53, 0, False),     # H*W*3 % 16 != 0: byte staging, byte stores, a short last chunk of 1961 % 16 = 9 pixels
    (40, 56, 5, False),     # a track base that is not 16-byte aligned
    (37, 53, 0, True),      # taps from global memory (LSD_WARP_L2_TAPS)
    (300, 300, 0, False),   # 270 KB frames: too large for shared memory, the global-tap variant by size
])
def test_warp_windows_bytes(model, H, W, offset, l2, monkeypatch):
    """The builder's output (lsd_warp_windows) equals the oracle byte for byte on geometries the model is not run on, covering
    every branch of the kernel: row-wrapping pixel chunks, the short tail, byte and 16-byte stores, both staging routes and both
    tap routes."""
    if l2:
        monkeypatch.setenv("LSD_WARP_L2_TAPS", "1")
    T, n_frames = 4, 11
    g = torch.Generator().manual_seed(H * W + offset)
    data = torch.randint(0, 256, (n_frames * H * W * 3 + 16,), generator=g, dtype=torch.uint8).cuda()
    track = data[offset:offset + n_frames * H * W * 3].view(n_frames, H, W, 3)
    ssr = P.shift_scale_rotate_warp
    mats = np.stack([np.broadcast_to(ssr(H, W, dx=-7.3, dy=5.6, scale=0.9, angle_deg=11), (T, 2, 3)),
                     np.broadcast_to(P.flip_warp(W), (T, 2, 3)), P.jitter_warps(T, H, W, 2.0, 0.05, 3)])
    starts = [0, 3, 7]
    p = lb.Predictor(model, chunk_size=T)
    n0 = model.launch_count()
    out = p.warp_track_windows(track, starts, mats).cpu().numpy()
    assert model.launch_count() == n0 + 1
    host = track.cpu().numpy()
    for i, s in enumerate(starts):
        for k in range(len(mats)):
            assert np.array_equal(out[i, k], wo.warp_window(host[s:s + T], mats[k])), (i, k)


@pytest.mark.gpu
def test_warp_windows_match_scored_rows(model):
    """The windows lsd_warp_windows returns are the ones lsd_score_warps scores: scored as a plain track they give its logits."""
    model.compute_precision = "bf16"
    track, mel = _track(65, n_frames=120)
    starts = [0, 50, 88]
    p = lb.Predictor(model, batch_size=16)
    mats = _variants(32, 96, 96)[:5]
    wins = p.warp_track_windows(track, starts, mats)
    flat = wins.reshape(-1, 96, 96, 3)
    a = [p._audio_start(s, 800, 120, 128) for s in starts for _ in mats]
    ref = _score_windows_explicit(p, flat, [r * 32 for r in range(len(starts) * len(mats))], mel, 120, a, 128).view(len(starts), -1)
    assert torch.equal(p.score_track_warps(track, starts, mel, 120, mats).cpu(), ref)


@pytest.mark.gpu
def test_warps_second_geometry(model):
    """T=16 windows of 64x64 crops, 64 mel columns, bf16, per-frame matrices."""
    model.compute_precision = "bf16"
    track, mel = _track(63, n_frames=120, H=64, W=64, Ta_full=480)
    n_frames = 120
    starts = [0, 9, 40, 77, 104]
    p = lb.Predictor(model, chunk_size=16, batch_size=8)
    mats = _variants(16, 64, 64)
    out = p.score_track_warps(track, starts, mel, n_frames, mats, chunk_a_size=64).cpu()
    ref = _host_reference(p, track, starts, mel, n_frames, mats, chunk_a_size=64)
    assert torch.equal(out, ref)


@pytest.mark.gpu
def test_warps_argument_errors(model):
    """Bad arguments return their status before anything is launched."""
    model.compute_precision = "bf16"
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8, device="cuda")
    mel = torch.zeros((1, 80, 300), device="cuda")
    p = lb.Predictor(model, batch_size=4)
    ident = P.shift_scale_rotate_warp(96, 96)
    n0 = model.launch_count()
    for w in (np.zeros((0, 2, 3)), np.stack([ident] * 65), np.zeros((1, 3, 3)), np.zeros((1, 31, 2, 3))):
        with pytest.raises(ValueError):
            p.score_track_warps(track, [0, 8], mel, 64, w)
    with pytest.raises(ValueError):
        p.score_track_warps(track, [0, 40], mel, 64, ident[None])        # window [40, 72) outside the 64-frame track
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    ws = model._workspace(1 << 20, track.device)
    out = torch.empty(2, 2, device="cuda")

    def call(mats, K, starts=(0, 8)):
        wc = None
        if mats is not None:
            wc = (_cabi.LsdWarp * (max(K, 1) * 32))()                   # K = 0 still passes a valid pointer
            for k in range(min(K, len(mats))):
                for t in range(32):
                    wc[k * 32 + t].m[:] = [float(v) for v in np.asarray(mats[k]).reshape(6)]
        return L.lsd_score_warps(h.ptr, track.data_ptr(), 64, 96, 96, (C.c_int32 * 2)(*starts), None, 2, 32, mel.data_ptr(), 80, 300, 64,
                                 128, wc, K, _cabi.LSD_PREC_BF16, 2, out.data_ptr(), ws.data_ptr(), ws.numel(), None)

    nan = ident.copy(); nan[0, 2] = float("nan")
    inf = ident.copy(); inf[1, 1] = float("inf")
    singular = np.array([[1.0, 2.0, 0.0], [2.0, 4.0, 0.0]])
    far = P.shift_scale_rotate_warp(96, 96, dx=-40000.0)             # its inverse maps pixels beyond 32767
    tiny = P.shift_scale_rotate_warp(96, 96, scale=1e-3)             # inverse scale 1000: 95 px * 1000 leaves the int16 range
    assert call(None, 1) == _cabi.LSD_ERR_ARG
    assert call([ident], 0) == _cabi.LSD_ERR_SHAPE
    assert call([ident] * 65, 65) == _cabi.LSD_ERR_SHAPE
    assert call([ident, nan], 2) == _cabi.LSD_ERR_ARG
    assert call([inf], 1) == _cabi.LSD_ERR_ARG
    assert call([singular], 1) == _cabi.LSD_ERR_ARG
    assert call([ident, far], 2) == _cabi.LSD_ERR_SHAPE
    assert call([tiny], 1) == _cabi.LSD_ERR_SHAPE
    assert call([ident], 1, starts=(0, 33)) == _cabi.LSD_ERR_SHAPE
    with pytest.raises(RuntimeError):
        p.score_track_warps(track, [0, 8], mel, 64, singular[None])
    assert model.launch_count() == n0


@pytest.mark.gpu
def test_robustness_track_matches_its_logits(model):
    model.compute_precision = "bf16"
    track, mel = _track(64)
    n_frames = 200
    starts = list(range(0, 169, 24))                                   # 8 windows
    p = lb.Predictor(model, batch_size=64)
    rb = p.robustness_track(track, starts, mel, n_frames, confidence_threshold=0.5)
    names, mats = P.robustness_variants(32, 96, 96)
    assert rb["variants"] == names and len(names) == 12 and rb["window_starts"] == starts
    logits = p.score_track_warps(track, starts, mel, n_frames, mats).cpu().numpy()
    probs = np.array([[p._calibrate(float(x)) for x in row] for row in logits])
    want = augmentation_stability(probs, 0.5, p.confidence_smoothing, p.trim_ratio)
    for k, v in want.items():
        assert np.array_equal(np.asarray(rb[k]), np.asarray(v)), k
    plain = [p._calibrate(float(x)) for x in p.score_track_logits(track, starts, mel, n_frames).cpu().tolist()]
    assert rb["confidence"] == p._robust_confidence(plain)


@pytest.mark.gpu
def test_long_video_robustness_entry_on_gpu(model):
    """robustness=True: `confidence` is the selected track's plain window aggregate, every other result key is unchanged."""
    model.compute_precision = "bf16"
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(model, batch_size=16)
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, robustness=True)
    assert set(res) == set(base) | {"robustness"}
    rb = res["robustness"]
    sel = next(t for t in res["tracks"] if t["track_id"] == res["selected_track_id"])
    assert rb["track_id"] == res["selected_track_id"]
    assert rb["confidence"] == pred._robust_confidence(sel["window_confidences"])
    tr = next(t for t in tracks if int(t["track_id"]) == rb["track_id"])
    assert rb["window_starts"] == [int(s) for s in tr["chunk_starts"]]   # absolute video frames
    assert len(rb["window_spread"]) == len(tr["chunk_starts"]) and len(rb["variant_confidence"]) == 12
    for k in base:
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k


# ---------------------------------------------------------------------------------------------------------------- CPU
def _cv2_warp(cv2, src, M):
    H, W = src.shape[:2]
    return cv2.warpAffine(src, np.asarray(M, dtype=np.float64), (W, H), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)


def test_oracle_matches_cv2_every_subpixel_shift():
    """The 1024 shifts (k/32, l/32) reach every entry of the weight table."""
    cv2 = pytest.importorskip("cv2")
    src = np.random.default_rng(0).integers(0, 256, (96, 96, 3), dtype=np.uint8)
    for k in range(32):
        for l in range(32):
            M = np.array([[1.0, 0.0, k / 32], [0.0, 1.0, l / 32]])
            assert np.array_equal(wo.warp_affine(src, M), _cv2_warp(cv2, src, M)), (k, l)


@pytest.mark.parametrize("H,W", [(96, 96), (64, 80)])
def test_oracle_matches_cv2_geometries(H, W):
    """Flips, rotations up to +-15 degrees, scales 0.8 - 1.25 and shifts that push taps past every border, square and not."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(H * W)
    src = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    mats = [P.flip_warp(W), np.array([[1.0, 0.0, 0.0], [0.0, -1.0, H - 1.0]]), np.array([[-1.0, 0.0, W - 1.0], [0.0, -1.0, H - 1.0]])]
    for dx, dy in [(30, 0), (-30, 0), (0, 30), (0, -30), (25.3, -28.9), (-29.5, 27.75)]:
        mats.append(P.shift_scale_rotate_warp(H, W, dx, dy))
    for _ in range(40):
        mats.append(P.shift_scale_rotate_warp(H, W, *rng.uniform(-30, 30, 2), rng.uniform(0.8, 1.25), rng.uniform(-15, 15)))
    for M in mats:
        assert np.array_equal(wo.warp_affine(src, M), _cv2_warp(cv2, src, M)), M
        assert np.array_equal(wo.invert_affine(M), cv2.invertAffineTransform(M)), M   # pins the inversion order bit for bit


def test_oracle_weight_table_closed_form():
    fy, fx = np.meshgrid(np.arange(32), np.arange(32), indexing="ij")
    closed = 32 * np.stack([(32 - fy) * (32 - fx), (32 - fy) * fx, fy * (32 - fx), fy * fx], axis=-1)
    assert np.array_equal(wo.TAB, closed)                              # the form warp_windows_kernel computes
    assert (wo.TAB.sum(axis=-1) == 32768).all()


def test_warp_window_per_frame():
    src = np.random.default_rng(3).integers(0, 256, (4, 16, 16, 3), dtype=np.uint8)
    mats = P.jitter_warps(4, 16, 16, 1.5, 0.02, 0)
    out = wo.warp_window(src, mats)
    assert out.shape == src.shape
    for t in range(4):
        assert np.array_equal(out[t], wo.warp_affine(src[t], mats[t]))
    assert np.array_equal(wo.warp_window(src, P.shift_scale_rotate_warp(16, 16)), src)   # the identity copies


def test_matrix_helpers_match_cv2():
    cv2 = pytest.importorskip("cv2")
    for H, W, dx, dy, s, a in [(96, 96, 0, 0, 1, 0), (96, 96, 4, -4, 0.92, 6), (64, 80, -2.5, 3.25, 1.08, -6), (64, 80, 0, 0, 1.25, 15)]:
        want = cv2.getRotationMatrix2D(((W - 1) / 2, (H - 1) / 2), a, s)
        want[0, 2] += dx
        want[1, 2] += dy
        assert np.abs(P.shift_scale_rotate_warp(H, W, dx, dy, s, a) - want).max() <= 1e-12
    src = np.random.default_rng(1).integers(0, 256, (64, 80, 3), dtype=np.uint8)
    assert np.array_equal(_cv2_warp(cv2, src, P.flip_warp(80)), cv2.flip(src, 1))


def test_jitter_and_default_variants():
    a, b = P.jitter_warps(32, 96, 96, 1.5, 0.02, 0), P.jitter_warps(32, 96, 96, 1.5, 0.02, 0)
    assert a.shape == (32, 2, 3) and np.array_equal(a, b)
    assert not np.array_equal(a, P.jitter_warps(32, 96, 96, 1.5, 0.02, 1))
    assert np.allclose(P.jitter_warps(8, 96, 96, 0.0, 0.0, 5), P.shift_scale_rotate_warp(96, 96))
    scale = np.hypot(a[:, 0, 0], a[:, 0, 1])
    assert np.allclose(a[:, 0, 0], a[:, 1, 1]) and np.allclose(a[:, 0, 1], 0) and 0.9 < scale.min() and scale.max() < 1.1
    names, mats = P.robustness_variants(32, 96, 96)
    assert names == ["identity", "flip", "shift_x+4", "shift_x-4", "shift_y+4", "shift_y-4", "scale_0.92", "scale_1.08", "rotate+6",
                     "rotate-6", "jitter_0", "jitter_1"]
    assert mats.shape == (12, 32, 2, 3)
    assert np.array_equal(mats[0, 5], np.array([[1.0, 0, 0], [0, 1.0, 0]]))
    assert np.array_equal(mats[2, 0], [[1.0, 0, 4], [0, 1.0, 0]]) and np.array_equal(mats[5, 0], [[1.0, 0, 0], [0, 1.0, -4]])
    assert np.array_equal(mats[10], P.jitter_warps(32, 96, 96, 1.5, 0.02, 0))


def test_augmentation_stability_hand_computed():
    # 4 windows x 3 variants (identity first), median aggregation, threshold 0.5
    p = [[0.60, 0.70, 0.40],
         [0.80, 0.75, 0.45],
         [0.30, 0.55, 0.20],
         [0.90, 0.85, 0.10]]
    r = augmentation_stability(p, 0.5, "median", 0.1)
    assert r["confidence"] == pytest.approx(0.70)                      # median(0.6, 0.8, 0.3, 0.9)
    assert r["variant_confidence"] == pytest.approx([0.70, 0.725, 0.30])
    assert r["tta_confidence"] == pytest.approx(np.median([1.70 / 3, 2.00 / 3, 1.05 / 3, 1.85 / 3]))
    assert np.allclose(r["window_spread"], [0.30, 0.35, 0.35, 0.80])
    # decisions differ from the identity's at (0,2), (1,2), (2,1), (3,2): 4 of 12
    assert r["decision_flip_rate"] == pytest.approx(4 / 12)
    assert r["verdict_stable"] is False                                # variant 2 aggregates to fake, the identity to real
    r = augmentation_stability([row[:2] for row in p], 0.5, "median", 0.1)
    assert r["verdict_stable"] is True and r["decision_flip_rate"] == pytest.approx(1 / 8)
    r = augmentation_stability(p, 0.5, "none", 0.1)
    assert r["confidence"] == pytest.approx(0.65) and r["variant_confidence"][2] == pytest.approx(0.2875)
    with pytest.raises(ValueError):
        augmentation_stability([0.5, 0.6])


def test_long_video_robustness_entry():
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def robustness_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"confidence": 0.7, "verdict_stable": True, "window_starts": [int(s) for s in tr["chunk_starts"]]}

    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, robustness=True, robustness_fn=robustness_fn,
                                            **fns)
    assert "robustness" not in base
    assert set(res) == set(base) | {"robustness"}
    assert res["robustness"]["track_id"] == res["selected_track_id"] == seen[0] and len(seen) == 1
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k
