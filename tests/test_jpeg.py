"""Compression robustness: `Predictor.score_track_jpeg` (lsd_score_jpeg), `Predictor.jpeg_track_windows` (lsd_jpeg_windows),
`Predictor.compression_track`, `aggregate.lowest_stable_quality` and the `compression` entry of `predict_long_video_from_tracks`.
The recompression is cv2's baseline JPEG encode + decode: oracle/jpeg_oracle.py restates it and is checked against cv2 here; the
logit of (window, variant) must be bit for bit the plain forward's logit for that window round-tripped on the host by the oracle."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import augmentation_stability, lowest_stable_quality
from oracle import jpeg_oracle as jo
from tests.golden.long_video_synth import SCENARIOS, make_audio, make_tracks

P = lb.Predictor
VARIANTS = [(None, None), (95, "420"), (75, "420"), (30, "420"), (5, "420"), (90, "444"), (40, "444"), (1, "444")]


def _cv2_round_trip(cv2, frame, q, sampling, order="bgr"):
    params = [cv2.IMWRITE_JPEG_QUALITY, int(q)]
    if sampling == "444":
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]
    bgr = cv2.cvtColor(frame, cv2.COLOR_RGB2BGR) if order == "rgb" else frame
    ok, buf = cv2.imencode(".jpg", bgr, params)
    assert ok
    out = cv2.imdecode(buf, cv2.IMREAD_COLOR)
    return cv2.cvtColor(out, cv2.COLOR_BGR2RGB) if order == "rgb" else out


def _smooth(rng, H, W, noise):
    import cv2
    base = cv2.resize(rng.integers(0, 256, (H // 8, W // 8, 3), dtype=np.uint8), (W, H), interpolation=cv2.INTER_CUBIC)
    return np.clip(base.astype(np.int64) + rng.normal(0, noise, base.shape), 0, 255).astype(np.uint8)


def _hard(rng, H, W):
    """Saturated 0 / 255 patches and hard colour edges: reaches the range limit of the inverse DCT and the output clamps."""
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    img[: H // 2, : W // 3] = (255, 0, 0)
    img[H // 2:, : W // 3] = (0, 0, 255)
    img[:, W // 3: W // 2] = 255
    img[H // 4: 3 * H // 4, W // 2: 3 * W // 4] = 0
    img[::2, 3 * W // 4:] = (0, 255, 255)
    img[1::2, 3 * W // 4:] = (255, 0, 255)
    return img


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("sampling", ["420", "444"])
def test_oracle_matches_cv2_every_quality(sampling):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(1 if sampling == "420" else 2)
    for q in range(1, 101):
        img = rng.integers(0, 256, (96, 96, 3), dtype=np.uint8) if q % 2 else _smooth(rng, 96, 96, q % 17)
        assert np.array_equal(jo.round_trip(img, q, sampling, "bgr"), _cv2_round_trip(cv2, img, q, sampling)), q


@pytest.mark.parametrize("H,W", [(64, 80), (112, 96)])
@pytest.mark.parametrize("sampling", ["420", "444"])
def test_oracle_matches_cv2_shapes_and_content(H, W, sampling):
    """Random, smooth and saturated / hard-edged crops at non-square sizes, in both channel orders."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(H * W + len(sampling))
    for q in (1, 5, 15, 30, 50, 51, 75, 90, 95, 100):
        for img in (rng.integers(0, 256, (H, W, 3), dtype=np.uint8), _smooth(rng, H, W, 4), _hard(rng, H, W)):
            for order in ("bgr", "rgb"):
                assert np.array_equal(jo.round_trip(img, q, sampling, order), _cv2_round_trip(cv2, img, q, sampling, order)), (q, order)


def test_oracle_rgb_is_cvtcolor_around_bgr():
    """The colour transform is not symmetric in R and B: an RGB frame gives a different result than the same bytes read as BGR."""
    img = _hard(np.random.default_rng(5), 96, 96)
    rgb = jo.round_trip(img, 50, "420", "rgb")
    assert np.array_equal(rgb, jo.round_trip_bgr(img[..., ::-1], 50, "420")[..., ::-1])
    assert not np.array_equal(rgb, jo.round_trip(img, 50, "420", "bgr"))
    assert np.array_equal(jo.round_trip(img, 50, None), img)


def test_oracle_int32_assertion_is_active():
    with pytest.raises(AssertionError):
        jo._i32(np.array([1 << 31]))
    jo._i32(np.array([(1 << 31) - 1, -(1 << 31)]))


ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
                   28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61,
                   54, 47, 55, 62, 63])


def _dqt_tables(buf: bytes):
    """{table id: (8, 8) natural-order table} from the DQT segments of a JPEG file (8-bit precision)."""
    tabs, i = {}, 2
    while i < len(buf) and buf[i] == 0xFF:
        marker, length = buf[i + 1], int.from_bytes(buf[i + 2:i + 4], "big")
        if marker == 0xDB:
            j = i + 4
            while j < i + 2 + length:
                pq, tq = buf[j] >> 4, buf[j] & 15
                assert pq == 0
                nat = np.zeros(64, dtype=np.int64)
                nat[ZIGZAG] = np.frombuffer(buf[j + 1:j + 65], dtype=np.uint8)
                tabs[tq] = nat.reshape(8, 8)
                j += 65
        if marker == 0xDA:
            break
        i += 2 + length
    return tabs


def test_quality_tables_match_cv2_files():
    cv2 = pytest.importorskip("cv2")
    img = np.random.default_rng(0).integers(0, 256, (16, 16, 3), dtype=np.uint8)
    for q in range(1, 101):
        tabs = _dqt_tables(cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])[1].tobytes())
        assert np.array_equal(tabs[0], jo.quality_table(jo.LUMA, q)), q
        assert np.array_equal(tabs[1], jo.quality_table(jo.CHROMA, q)), q


def test_lowest_stable_quality_hand_computed():
    qs = [None, 95, 85, 75, 60, 45, 30, 15]
    # plain 0.8 (real), threshold 0.5
    assert lowest_stable_quality(qs, [0.8, 0.8, 0.7, 0.7, 0.6, 0.55, 0.51, 0.5], 0.8, 0.5) == 15       # all stable
    assert lowest_stable_quality(qs, [0.8, 0.49, 0.7, 0.7, 0.6, 0.6, 0.6, 0.6], 0.8, 0.5) is None      # q95 flips
    assert lowest_stable_quality(qs, [0.8, 0.7, 0.7, 0.6, 0.4, 0.6, 0.3, 0.2], 0.8, 0.5) == 75         # flip at q60
    # non-monotone: q85 flips, q75 and below are back on the plain side; the flip at 85 hides them
    assert lowest_stable_quality(qs, [0.8, 0.7, 0.4, 0.7, 0.7, 0.7, 0.7, 0.7], 0.8, 0.5) == 95
    # a fake plain verdict: the side is "below the threshold"
    assert lowest_stable_quality(qs, [0.2, 0.3, 0.4, 0.49, 0.5, 0.3, 0.3, 0.3], 0.2, 0.5) == 75
    # two variants at one quality (4:2:0 and 4:4:4): both must hold
    assert lowest_stable_quality([None, 90, 90, 50], [0.8, 0.9, 0.3, 0.9], 0.8, 0.5) is None
    assert lowest_stable_quality([None], [0.8], 0.8, 0.5) is None
    with pytest.raises(ValueError):
        lowest_stable_quality([95, 85], [0.5], 0.5)


def test_default_compression_variants():
    names, variants = P.compression_variants()
    assert names == ["none", "q95", "q85", "q75", "q60", "q45", "q30", "q15"]
    assert variants == [(None, None)] + [(q, "420") for q in (95, 85, 75, 60, 45, 30, 15)]


@pytest.mark.parametrize("H,W,variants", [
    (88, 96, [(50, "420")]),                      # H not a multiple of 16 with 4:2:0
    (96, 100, [(50, "444")]),                     # W not a multiple of 8
    (96, 96, [(0, "420")]), (96, 96, [(101, "444")]),
    (96, 96, []), (96, 96, [(50, "420")] * 65),
    (96, 96, [(50, "422")]),
])
def test_argument_errors_raise_value_error(H, W, variants):
    pred = P(None, device=torch.device("cpu"))
    track = torch.zeros((40, H, W, 3), dtype=torch.uint8)
    mel = torch.zeros((1, 80, 200))
    with pytest.raises(ValueError):
        pred.score_track_jpeg(track, [0], mel, 40, variants)
    with pytest.raises(ValueError):
        pred.jpeg_track_windows(track, [0], variants)


def test_argument_errors_channel_order_and_window():
    pred = P(None, device=torch.device("cpu"))
    track = torch.zeros((40, 96, 96, 3), dtype=torch.uint8)
    with pytest.raises(ValueError):
        pred.jpeg_track_windows(track, [0], [(50, "420")], channel_order="yuv")
    with pytest.raises(ValueError):
        pred.jpeg_track_windows(track, [9], [(50, "420")])                     # window [9, 41) outside the 40-frame track
    # 88-pixel sides are fine for 4:4:4 alone
    assert pred._jpeg_args(torch.zeros((40, 88, 88, 3), dtype=torch.uint8), [0], [(50, "444"), (None, None)], "rgb")[0] == 2


def test_long_video_compression_entry():
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def compression_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"confidence": 0.7, "lowest_stable_quality": 45, "window_starts": [int(s) for s in tr["chunk_starts"]]}

    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, compression=True,
                                            compression_fn=compression_fn, **fns)
    assert "compression" not in base
    assert set(res) == set(base) | {"compression"}
    assert res["compression"]["track_id"] == res["selected_track_id"] == seen[0] and len(seen) == 1
    assert res["compression"]["lowest_stable_quality"] == 45
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k


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


def _host_reference(p, track, starts, mel, total_v_frames, variants, order="rgb", chunk_a_size=128):
    """(n, K) logits: every (window, variant) round-tripped by the oracle, the windows laid end to end as one track and scored by
    lsd_score_windows with the window's own audio start."""
    T = p.chunk_size
    host = track.cpu().numpy()
    wins = [jo.round_trip_window(host[s:s + T], q, smp, order) for s in starts for q, smp in variants]
    flat = torch.from_numpy(np.concatenate(wins)).cuda()
    a = [p._audio_start(s, int(mel.shape[2]), total_v_frames, chunk_a_size) for s in starts for _ in variants]
    ref = _score_windows_explicit(p, flat, [r * T for r in range(len(wins))], mel, total_v_frames, a, chunk_a_size)
    return ref.view(len(starts), len(variants))


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(96, 96), (64, 80)])
@pytest.mark.parametrize("order", ["rgb", "bgr"])
@pytest.mark.parametrize("offset", [0, 3])
def test_jpeg_windows_bytes(model, H, W, order, offset):
    """The builder's output (lsd_jpeg_windows) equals the oracle byte for byte: both samplings, qualities 1 to 95, the plain
    copy, both channel orders; offset 3: a track base that is not 16-byte aligned (byte loads and stores)."""
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
    out = p.jpeg_track_windows(track, starts, VARIANTS, channel_order=order).cpu().numpy()
    assert model.launch_count() == n0 + 1
    host = host.numpy()
    for i, s in enumerate(starts):
        for k, (q, smp) in enumerate(VARIANTS):
            assert np.array_equal(out[i, k], jo.round_trip_window(host[s:s + T], q, smp, order)), (i, k)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_jpeg_bitwise(model, prec):
    """Every (window, variant) logit equals the plain forward of the window round-tripped by the oracle, with explicit audio
    starts; the plain column equals score_track_logits."""
    model.compute_precision = prec
    track, mel = _track(71)
    n_frames = 200
    starts = list(range(0, n_frames - 32 + 1, 21))                   # 9 windows x 8 variants: 72 rows, 5 batches of 16
    p = lb.Predictor(model, batch_size=16)
    a_from = [s + 3 for s in starts]
    out = p.score_track_jpeg(track, starts, mel, n_frames, VARIANTS, audio_starts_from=a_from).cpu()
    assert out.shape == (len(starts), len(VARIANTS)) and out.dtype == torch.float32
    T = 32
    host = track.cpu().numpy()
    wins = [jo.round_trip_window(host[s:s + T], q, smp, "rgb") for s in starts for q, smp in VARIANTS]
    flat = torch.from_numpy(np.concatenate(wins)).cuda()
    a = [p._audio_start(v, 800, n_frames, 128) for v in a_from for _ in VARIANTS]
    ref = _score_windows_explicit(p, flat, [r * T for r in range(len(wins))], mel, n_frames, a, 128).view(len(starts), -1)
    assert torch.equal(out, ref)
    plain = p.score_track_jpeg(track, starts, mel, n_frames, VARIANTS)[:, 0].cpu()
    assert torch.equal(plain, p.score_track_logits(track, starts, mel, n_frames).cpu())
    assert not torch.equal(out[:, 4], out[:, 0])


def _jpeg_raw(model, track, starts, mel, n_frames, variants, batch, ws_bytes, order=_cabi.LSD_RGB, T=32, Ta=128):
    """lsd_score_jpeg straight through the C-ABI, in a workspace of exactly ws_bytes, twice on the same workspace."""
    L = _cabi.lib()
    n, K = len(starts), len(variants)
    H, W = int(track.shape[1]), int(track.shape[2])
    smp = {None: _cabi.LSD_JPEG_NONE, "444": _cabi.LSD_JPEG_444, "420": _cabi.LSD_JPEG_420}
    vc = (_cabi.LsdJpeg * K)(*[_cabi.LsdJpeg(q or 0, smp[s]) for q, s in variants])
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        L.lsd_workspace_invalidate(h.ptr)
        logits = torch.empty(n, K, dtype=torch.float32, device="cuda")
        for _ in range(2):
            rc = L.lsd_score_jpeg(h.ptr, track.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*starts), None, n, T, mel.data_ptr(),
                                  int(mel.shape[1]), int(mel.shape[2]), n_frames, Ta, vc, K, order, model._precision(), batch,
                                  logits.data_ptr(), ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
            _cabi.check(h.ptr, rc)
            out = logits.cpu()
        L.lsd_workspace_invalidate(h.ptr)
    return out


@pytest.mark.gpu
def test_jpeg_batches_and_exact_workspace(model):
    """batch=7 over 54 rows (7 full batches and a short one of 5): pipelined in a double workspace and again in exactly the queried
    workspace, both equal to one batch of 64 and to the host reference."""
    model.compute_precision = "bf16"
    track, mel = _track(72)
    n_frames = 200
    starts = list(range(0, 169, 21))                                  # 9 windows
    variants = VARIANTS[1:7]                                          # K = 6
    L = _cabi.lib()
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        need7 = L.lsd_score_jpeg_workspace_bytes(h.ptr, 7, 6, 32, 96, 96, 80, 128, _cabi.LSD_PREC_BF16)
        need64 = L.lsd_score_jpeg_workspace_bytes(h.ptr, 64, 6, 32, 96, 96, 80, 128, _cabi.LSD_PREC_BF16)
    assert 0 < need7 < need64
    one = _jpeg_raw(model, track, starts, mel, n_frames, variants, 64, need64)
    piped = _jpeg_raw(model, track, starts, mel, n_frames, variants, 7, 2 * need7)
    exact = _jpeg_raw(model, track, starts, mel, n_frames, variants, 7, need7)
    assert torch.equal(piped, one) and torch.equal(exact, one)
    p = lb.Predictor(model, batch_size=64)
    assert torch.equal(one, _host_reference(p, track, starts, mel, n_frames, variants))
    bgr = _jpeg_raw(model, track, starts, mel, n_frames, variants, 7, 2 * need7, order=_cabi.LSD_BGR)
    assert torch.equal(bgr, _host_reference(p, track, starts, mel, n_frames, variants, order="bgr"))


@pytest.mark.gpu
def test_jpeg_argument_errors(model):
    """Bad arguments return their status before anything is launched."""
    model.compute_precision = "bf16"
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8, device="cuda")
    mel = torch.zeros((1, 80, 300), device="cuda")
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    ws = model._workspace(1 << 20, track.device)
    out = torch.empty(2, 2, device="cuda")
    n0 = model.launch_count()

    def call(variants, K=None, starts=(0, 8), order=_cabi.LSD_RGB, HW=(96, 96), null=False):
        K = len(variants) if K is None else K
        vc = None if null else (_cabi.LsdJpeg * max(K, 1))(*[_cabi.LsdJpeg(q, s) for q, s in variants][:max(K, 1)])
        rc = L.lsd_score_jpeg(h.ptr, track.data_ptr(), 64, HW[0], HW[1], (C.c_int32 * 2)(*starts), None, 2, 32, mel.data_ptr(), 80, 300,
                              64, 128, vc, K, order, _cabi.LSD_PREC_BF16, 2, out.data_ptr(), ws.data_ptr(), ws.numel(), None)
        wrc = L.lsd_jpeg_windows(h.ptr, track.data_ptr(), 64, HW[0], HW[1], (C.c_int32 * 2)(*starts), 2, 32, vc, K, order, out.data_ptr(),
                                 ws.data_ptr(), ws.numel(), None)
        assert wrc == rc
        return rc

    ok = (50, _cabi.LSD_JPEG_420)
    assert call([ok], null=True) == _cabi.LSD_ERR_ARG
    assert call([ok], K=0) == _cabi.LSD_ERR_SHAPE
    assert call([ok] * 65) == _cabi.LSD_ERR_SHAPE
    assert call([ok, (0, _cabi.LSD_JPEG_420)]) == _cabi.LSD_ERR_ARG
    assert call([(101, _cabi.LSD_JPEG_444)]) == _cabi.LSD_ERR_ARG
    assert call([(50, 3)]) == _cabi.LSD_ERR_ARG
    assert call([ok], order=2) == _cabi.LSD_ERR_ARG
    assert call([ok], HW=(88, 96)) == _cabi.LSD_ERR_SHAPE                  # 4:2:0 needs multiples of 16
    assert call([(50, _cabi.LSD_JPEG_444)], HW=(96, 92)) == _cabi.LSD_ERR_SHAPE
    assert call([ok], HW=(256, 256)) == _cabi.LSD_ERR_SHAPE                # the planes do not fit in shared memory
    assert call([ok], starts=(0, 33)) == _cabi.LSD_ERR_SHAPE               # window [33, 65) outside the 64-frame track
    assert call([(0, _cabi.LSD_JPEG_NONE)], starts=(0, 33)) == _cabi.LSD_ERR_SHAPE   # quality unused for the plain copy
    assert model.launch_count() == n0


@pytest.mark.gpu
def test_compression_track_matches_its_logits(model):
    model.compute_precision = "bf16"
    track, mel = _track(73)
    n_frames = 200
    starts = list(range(0, 169, 24))                                   # 8 windows
    p = lb.Predictor(model, batch_size=64)
    ct = p.compression_track(track, starts, mel, n_frames, confidence_threshold=0.5)
    names, variants = P.compression_variants()
    assert ct["variants"] == names and ct["qualities"] == [q for q, _ in variants] and ct["window_starts"] == starts
    logits = p.score_track_jpeg(track, starts, mel, n_frames, variants).cpu().numpy()
    probs = np.array([[p._calibrate(float(x)) for x in row] for row in logits])
    want = augmentation_stability(probs, 0.5, p.confidence_smoothing, p.trim_ratio)
    for k, v in want.items():
        assert np.array_equal(np.asarray(ct[k]), np.asarray(v)), k
    assert ct["lowest_stable_quality"] == lowest_stable_quality(ct["qualities"], want["variant_confidence"], want["confidence"], 0.5)
    plain = [p._calibrate(float(x)) for x in p.score_track_logits(track, starts, mel, n_frames).cpu().tolist()]
    assert ct["confidence"] == p._robust_confidence(plain)


@pytest.mark.gpu
def test_long_video_compression_entry_on_gpu(model):
    """compression=True: `confidence` is the selected track's plain window aggregate, every other result key is unchanged."""
    model.compute_precision = "bf16"
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(model, batch_size=16)
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, compression=True)
    assert set(res) == set(base) | {"compression"}
    cp = res["compression"]
    sel = next(t for t in res["tracks"] if t["track_id"] == res["selected_track_id"])
    assert cp["track_id"] == res["selected_track_id"]
    assert cp["confidence"] == pred._robust_confidence(sel["window_confidences"])
    tr = next(t for t in tracks if int(t["track_id"]) == cp["track_id"])
    assert cp["window_starts"] == [int(s) for s in tr["chunk_starts"]]
    assert len(cp["variant_confidence"]) == 8
    for k in base:
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k
