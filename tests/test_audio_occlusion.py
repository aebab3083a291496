"""Audio occlusion evidence: `Predictor.score_track_audio_occlusions` (lsd_score_audio_occlusions), the box helpers,
`Predictor.explain_track_audio`, `aggregate.columns_to_frames` and the `audio_evidence` entry of `predict_long_video_from_tracks`.
The logit of (window, box) must be bit for bit the plain forward's logit for that window with its log-mel slice masked on the host."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import columns_to_frames, frame_evidence_timeline
from tests.golden.long_video_synth import SCENARIOS, make_audio, make_tracks

# (c0, c1, f0, f1) for 128-column, 80-bin slices
BOXES = [
    (0, 0, 0, 0),          # empty: the plain window
    (0, 16, 0, 80),        # full-height time segment at the start ...
    (48, 64, 0, 80),       # ... and in the middle
    (0, 128, 0, 10),       # full-width band at the bottom ...
    (0, 128, 70, 80),      # ... and one touching bin F
    (100, 128, 20, 50),    # touches column Ta
    (37, 38, 0, 80),       # one column
    (0, 128, 41, 42),      # one bin
    (5, 90, 13, 61),       # an inner rectangle
]


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()


@pytest.fixture(scope="module")
def model(built, seed0_sd):
    m = lb.LipSyncModel()
    m.load_state_dict(seed0_sd, strict=True)
    return m.to("cuda:0").eval()


def _mask(win, box, fill):
    """numpy statement of the box rule on one (F, Ta) log-mel slice."""
    c0, c1, f0, f1 = box
    out = win.copy()
    out[f0:f1, c0:c1] = fill
    return out


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
                                 (C.c_int32 * n)(*[int(s) for s in starts]), (C.c_int32 * n)(*[int(x) for x in a_starts]), n, p.chunk_size,
                                 mel.data_ptr(), int(mel.shape[1]), int(mel.shape[2]), total_v_frames, chunk_a_size, prec, batch,
                                 out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
        _cabi.check(h.ptr, rc)
    return out.cpu()


def _host_reference(p, track, starts, mel, total_v_frames, boxes, fill, chunk_a_size=128):
    """(n, K) logits: every window's slice (`_align_audio_chunk`) masked by every box with numpy, the n*K masked slices laid end to
    end as one (1, F, n*K*Ta) clip and scored by lsd_score_windows, each window's start repeated K times, audio starts r*Ta."""
    Ta = chunk_a_size
    host = mel.cpu().numpy()
    slices = [_mask(p._align_audio_chunk(host, s, total_v_frames, Ta)[0], b, fill) for s in starts for b in boxes]
    clip = torch.from_numpy(np.concatenate(slices, axis=1)[None]).cuda()
    vs = [s for s in starts for _ in boxes]
    ref = _score_windows_explicit(p, track, vs, clip, total_v_frames, [r * Ta for r in range(len(slices))], Ta)
    return ref.view(len(starts), len(boxes))


def _track(seed, n_frames=200, H=96, W=96, Ta_full=800):
    g = torch.Generator().manual_seed(seed)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    mel = (-80.0 * torch.rand((1, 80, Ta_full), generator=g)).cuda()
    return track, mel


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_audio_occlusions_bitwise(model, prec):
    """Every (window, box) logit equals the plain forward of the host-masked slice; the empty box equals score_track_logits."""
    model.compute_precision = prec
    track, mel = _track(61)
    n_frames = 200
    starts = list(range(0, n_frames - 32 + 1, 21))                   # 9 windows in batches of 4, 4 and 1
    p = lb.Predictor(model, batch_size=4)
    out = p.score_track_audio_occlusions(track, starts, mel, n_frames, BOXES, fill=-37.5).cpu()
    assert out.shape == (len(starts), len(BOXES)) and out.dtype == torch.float32
    ref = _host_reference(p, track, starts, mel, n_frames, BOXES, -37.5)
    for k in range(len(BOXES)):
        assert torch.equal(out[:, k], ref[:, k]), (k, out[:, k], ref[:, k])
    assert torch.equal(out[:, 0], p.score_track_logits(track, starts, mel, n_frames).cpu())
    assert not torch.equal(out[:, 1], out[:, 0])                      # the mask changed something


def _audio_occlusions_raw(model, track, starts, mel, n_frames, boxes, fill, batch, ws_bytes, T=32, Ta=128):
    """lsd_score_audio_occlusions straight through the C-ABI, in a workspace of exactly ws_bytes (called twice: the second call
    reuses the zero padding of the first)."""
    L = _cabi.lib()
    n, K = len(starts), len(boxes)
    H, W = int(track.shape[1]), int(track.shape[2])
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        L.lsd_workspace_invalidate(h.ptr)
        logits = torch.empty(n, K, dtype=torch.float32, device="cuda")
        bc = (_cabi.LsdAudioOcclusion * K)(*[_cabi.LsdAudioOcclusion(*b) for b in boxes])
        for _ in range(2):
            rc = L.lsd_score_audio_occlusions(h.ptr, track.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*starts), None, n, T, mel.data_ptr(),
                                              int(mel.shape[1]), int(mel.shape[2]), n_frames, Ta, bc, K, fill, model._precision(), batch,
                                              logits.data_ptr(), ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
            _cabi.check(h.ptr, rc)
            out = logits.cpu()
        L.lsd_workspace_invalidate(h.ptr)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("misaligned", [False, True])
def test_audio_occlusions_groups_and_exact_workspace(model, monkeypatch, misaligned):
    """LSD_VARIANT_ROWS=20 and K = 9 give audio groups of 2 windows; 9 windows in batches of 5 end with a batch of 4 (groups 2 + 2),
    and batches of 3 have a shorter last group (2 + 1).  Every run, in exactly the queried workspace and called twice, equals one
    batch of 64 and the host reference.  misaligned: a track that is not 16-byte aligned takes the gather route."""
    monkeypatch.setenv("LSD_VARIANT_ROWS", "20")
    model.compute_precision = "bf16"
    n_frames, H, W = 200, 96, 96
    g = torch.Generator().manual_seed(62)
    data = torch.randint(0, 256, (n_frames * H * W * 3 + 16,), generator=g, dtype=torch.uint8).cuda()
    o = 1 if misaligned else 0
    track = data[o:o + n_frames * H * W * 3].view(n_frames, H, W, 3)
    mel = (-80.0 * torch.rand((1, 80, 800), generator=g)).cuda()
    starts = list(range(0, 169, 21))                                  # 9 windows
    K = len(BOXES)
    L = _cabi.lib()
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        need = {b: L.lsd_score_audio_occlusions_workspace_bytes(h.ptr, b, K, 32, H, W, 80, 128, _cabi.LSD_PREC_BF16) for b in (3, 5, 64)}
    assert 0 < need[3] < need[5] < need[64]
    one = _audio_occlusions_raw(model, track, starts, mel, n_frames, BOXES, -80.0, 64, need[64])
    for b in (3, 5):
        assert torch.equal(_audio_occlusions_raw(model, track, starts, mel, n_frames, BOXES, -80.0, b, need[b]), one), b
    p = lb.Predictor(model, batch_size=64)
    assert torch.equal(one, _host_reference(p, track.contiguous(), starts, mel, n_frames, BOXES, -80.0))


@pytest.mark.gpu
def test_audio_occlusions_second_geometry(model):
    """T=16 windows of 64x64 crops, 64 mel columns, bf16."""
    model.compute_precision = "bf16"
    track, mel = _track(63, n_frames=120, H=64, W=64, Ta_full=480)
    n_frames = 120
    starts = [0, 9, 40, 77, 104]
    p = lb.Predictor(model, chunk_size=16, batch_size=2)
    boxes = [(0, 0, 0, 0), (60, 64, 0, 80), (10, 11, 5, 79)] + p.mute_segment_boxes(64, 16) + p.mel_band_boxes(64, 80, 3)
    out = p.score_track_audio_occlusions(track, starts, mel, n_frames, boxes, chunk_a_size=64).cpu()
    ref = _host_reference(p, track, starts, mel, n_frames, boxes, -80.0, chunk_a_size=64)
    assert torch.equal(out, ref)


@pytest.mark.gpu
def test_audio_occlusions_fallback_route(model, monkeypatch):
    """The launch-by-launch token path (LSD_TOK_FRONT=0) scores the pseudo clip with lsd_score_windows: same bits as the reference."""
    monkeypatch.setenv("LSD_TOK_FRONT", "0")
    model.compute_precision = "bf16"
    track, mel = _track(64)
    n_frames = 200
    starts = [0, 50, 111, 168]
    p = lb.Predictor(model, batch_size=3)
    out = p.score_track_audio_occlusions(track, starts, mel, n_frames, BOXES).cpu()
    assert torch.equal(out, _host_reference(p, track, starts, mel, n_frames, BOXES, -80.0))


@pytest.mark.gpu
def test_audio_occlusions_short_clip(model):
    """A clip of 100 columns under 128-column slices: every slice starts at 0 and repeats column 99; masking applies after the
    padding, so a box over columns 100..127 masks repeated columns."""
    model.compute_precision = "bf16"
    track, mel = _track(65, n_frames=80, Ta_full=100)
    n_frames = 80
    starts = [0, 20, 48]
    p = lb.Predictor(model, batch_size=64)
    boxes = [(0, 0, 0, 0), (100, 128, 0, 80), (90, 110, 30, 60)]
    out = p.score_track_audio_occlusions(track, starts, mel, n_frames, boxes).cpu()
    assert torch.equal(out, _host_reference(p, track, starts, mel, n_frames, boxes, -80.0))
    assert not torch.equal(out[:, 1], out[:, 0])


@pytest.mark.gpu
def test_audio_occlusion_argument_errors(model):
    """Bad arguments raise ValueError (LSD_ERR_SHAPE / LSD_ERR_ARG at the C-ABI) before anything is launched."""
    model.compute_precision = "bf16"
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8, device="cuda")
    mel = torch.zeros((1, 80, 300), device="cuda")
    p = lb.Predictor(model, batch_size=4)
    good = [(0, 0, 0, 0)]
    bad_boxes = [[], good * 65, [(0, 129, 0, 80)], [(-1, 4, 0, 80)], [(5, 4, 0, 80)], [(0, 4, 10, 9)], [(0, 4, 0, 81)],
                 [(0, 4, -1, 80)], [(0, 4, 0)]]
    n0 = model.launch_count()
    for b in bad_boxes:
        with pytest.raises(ValueError):
            p.score_track_audio_occlusions(track, [0, 8], mel, 64, b)
    with pytest.raises(ValueError):
        p.score_track_audio_occlusions(track, [0, 40], mel, 64, good)    # window [40, 72) outside the 64-frame track
    for fill in (float("nan"), float("inf")):
        with pytest.raises(ValueError):
            p.score_track_audio_occlusions(track, [0], mel, 64, good, fill=fill)
    # the C-ABI itself
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    ws = model._workspace(1 << 20, track.device)
    out = torch.empty(2, 2, device="cuda")
    st = (C.c_int32 * 2)(0, 8)

    def call(boxes, K, fill=-80.0, starts=st, ws_bytes=ws.numel(), mel_ptr=mel.data_ptr()):
        return L.lsd_score_audio_occlusions(h.ptr, track.data_ptr(), 64, 96, 96, starts, None, 2, 32, mel_ptr, 80, 300, 64, 128,
                                            boxes, K, fill, _cabi.LSD_PREC_BF16, 2, out.data_ptr(), ws.data_ptr(), ws_bytes, None)

    one = (_cabi.LsdAudioOcclusion * 1)(_cabi.LsdAudioOcclusion(0, 0, 0, 0))
    many = (_cabi.LsdAudioOcclusion * 65)(*[_cabi.LsdAudioOcclusion(0, 0, 0, 0)] * 65)
    assert call(None, 1) == _cabi.LSD_ERR_ARG
    assert call(one, 0) == _cabi.LSD_ERR_SHAPE
    assert call(many, 65) == _cabi.LSD_ERR_SHAPE
    assert call(one, 1, fill=float("nan")) == _cabi.LSD_ERR_ARG
    assert call(one, 1, fill=float("-inf")) == _cabi.LSD_ERR_ARG
    assert call((_cabi.LsdAudioOcclusion * 1)(_cabi.LsdAudioOcclusion(0, 129, 0, 80)), 1) == _cabi.LSD_ERR_SHAPE
    assert call((_cabi.LsdAudioOcclusion * 1)(_cabi.LsdAudioOcclusion(0, 4, 50, 40)), 1) == _cabi.LSD_ERR_SHAPE
    assert call((_cabi.LsdAudioOcclusion * 1)(_cabi.LsdAudioOcclusion(0, 4, 0, 81)), 1) == _cabi.LSD_ERR_SHAPE
    assert call(one, 1, starts=(C.c_int32 * 2)(0, 33)) == _cabi.LSD_ERR_SHAPE
    assert call(one, 1, mel_ptr=None) == _cabi.LSD_ERR_ARG
    assert call(one, 1, ws_bytes=1024) == _cabi.LSD_ERR_WORKSPACE
    assert model.launch_count() == n0


@pytest.mark.gpu
def test_explain_track_audio_matches_its_logits(model):
    model.compute_precision = "bf16"
    track, mel = _track(66)
    n_frames = 200
    starts = list(range(0, 169, 24))                                   # 8 windows
    p = lb.Predictor(model, batch_size=64)
    ex = p.explain_track_audio(track, starts, mel, n_frames)
    S, nb, Ta = 8, 8, 128
    boxes = [(0, 0, 0, 0)] + p.mute_segment_boxes(Ta, 16) + p.mel_band_boxes(Ta, 80, 8)
    logits = p.score_track_audio_occlusions(track, starts, mel, n_frames, boxes).cpu().numpy()
    probs = np.array([[p._calibrate(float(x)) for x in row] for row in logits])
    assert np.array_equal(ex["confidence"], probs[:, 0])
    assert np.array_equal(ex["audio_temporal"], probs[:, 1:1 + S] - probs[:, :1])
    assert np.array_equal(ex["audio_spectral"], probs[:, 1 + S:] - probs[:, :1])
    assert np.allclose(ex["audio_spectral_mean"], ex["audio_spectral"].mean(axis=0))
    a = [p._audio_start(s, 800, n_frames) for s in starts]
    first, tl = frame_evidence_timeline(a, ex["audio_temporal"], 16, Ta)
    assert ex["column_first"] == first == 0 and ex["column_evidence"] == tl and len(tl) == a[-1] + Ta
    assert (ex["frame_first"], ex["frame_evidence"]) == columns_to_frames(first, tl, 800, n_frames)
    assert (ex["segment_cols"], ex["bands"], ex["band_edges"], ex["fill"]) == (16, 8, [0, 10, 20, 30, 40, 50, 60, 70, 80], -80.0)
    # the confidence column is the plain window score, and explain_track's
    assert np.array_equal(ex["confidence"], p.explain_track(track, starts, mel, n_frames)["confidence"])


@pytest.mark.gpu
def test_long_video_audio_evidence_entry_on_gpu(model):
    """audio_evidence=True: `confidence` equals the selected track's window confidences, every other result key is unchanged."""
    model.compute_precision = "bf16"
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(model, batch_size=16)
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, audio_evidence=True)
    assert set(res) == set(base) | {"audio_evidence"}
    ev = res["audio_evidence"]
    sel = next(t for t in res["tracks"] if t["track_id"] == res["selected_track_id"])
    assert ev["track_id"] == res["selected_track_id"]
    assert ev["confidence"].tolist() == sel["window_confidences"]
    tr = next(t for t in tracks if int(t["track_id"]) == ev["track_id"])
    Ta_full = int(np.asarray(mel).shape[-1])
    a = [pred._audio_start(int(s), Ta_full, n_frames) for s in tr["chunk_starts"]]
    assert ev["column_first"] == min(a)                                # absolute mel columns
    assert ev["column_first"] + len(ev["column_evidence"]) <= Ta_full
    assert ev["frame_first"] == min(a) * n_frames // Ta_full           # absolute video frames
    for k in base:
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_mute_segment_boxes():
    P = lb.Predictor
    b = P.mute_segment_boxes(128, 16)
    assert len(b) == 8 and b[0] == (0, 16, 0, 80) and b[7] == (112, 128, 0, 80)
    assert P.mute_segment_boxes(40, 16, 64) == [(0, 16, 0, 64), (16, 32, 0, 64), (32, 40, 0, 64)]
    assert P.mute_segment_boxes(10, 20) == [(0, 10, 0, 80)]
    cover = np.zeros(100, dtype=int)
    for c0, c1, _, _ in P.mute_segment_boxes(100, 7):
        cover[c0:c1] += 1
    assert (cover == 1).all()
    for s in (0, -3):
        with pytest.raises(ValueError):
            P.mute_segment_boxes(128, s)


def test_mel_band_boxes():
    P = lb.Predictor
    b = P.mel_band_boxes(128, 80, 8)
    assert len(b) == 8 and b[0] == (0, 128, 0, 10) and b[7] == (0, 128, 70, 80)
    assert [(f0, f1) for _, _, f0, f1 in P.mel_band_boxes(64, 10, 3)] == [(0, 3), (3, 7), (7, 10)]   # round(j*10/3)
    assert P.mel_band_boxes(16, 5, 5) == [(0, 16, j, j + 1) for j in range(5)]
    for g in (0, 81):
        with pytest.raises(ValueError):
            P.mel_band_boxes(128, 80, g)


def test_columns_to_frames_hand_computed():
    # 10 columns per frame: columns 25..44 -> frames 2 (25-29), 3 (30-39), 4 (40-44)
    first, v = columns_to_frames(25, [1.0] * 5 + [2.0] * 10 + [4.0, None, 6.0, None, None], 100, 10)
    assert first == 2 and v == pytest.approx([1.0, 2.0, 5.0])
    # Ta_full = 7, 3 frames: column c -> c * 3 // 7 = 0 0 0 1 1 2 2; a frame whose columns are all None has no value
    first, v = columns_to_frames(0, [1, 2, 3, None, None, 5, 7], 7, 3)
    assert first == 0 and v == [2.0, None, 6.0]
    # more frames than columns (Ta_full = 4, 10 frames): column c -> frame 0, 2, 5, 7; the frames between have no column
    first, v = columns_to_frames(0, [1, 2, 3, 4], 4, 10)
    assert first == 0 and v == [1.0, None, 2.0, None, None, 3.0, None, 4.0]
    assert columns_to_frames(5, [], 100, 10) == (0, [])
    with pytest.raises(ValueError):
        columns_to_frames(0, [1.0], 0, 10)


def test_long_video_audio_evidence_entry():
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def audio_evidence_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"confidence": np.full(len(tr["chunk_starts"]), 0.7), "column_first": 0}

    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, audio_evidence=True,
                                            audio_evidence_fn=audio_evidence_fn, **fns)
    assert "audio_evidence" not in base
    assert set(res) == set(base) | {"audio_evidence"}
    assert res["audio_evidence"]["track_id"] == res["selected_track_id"] == seen[0] and len(seen) == 1
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k
