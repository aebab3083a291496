"""Occlusion evidence: `Predictor.score_track_occlusions` (lsd_score_occlusions), the box helpers, `Predictor.explain_track`,
`aggregate.frame_evidence_timeline` and the `evidence` entry of `predict_long_video_from_tracks`.
The logit of (window, box) must be bit for bit the plain forward's logit for that window occluded on the host."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import frame_evidence_timeline
from tests.golden.long_video_synth import SCENARIOS, make_audio, make_tracks

# (t0, t1, y0, y1, x0, x1, src) for T = 32, 96 x 96 crops
BOXES = [
    (0, 0, 0, 0, 0, 0, -1),          # empty: the plain window
    (8, 12, 0, 96, 0, 96, 7),        # freeze from the frame before the segment
    (0, 4, 0, 96, 0, 96, 4),         # freeze from the frame after the segment
    (0, 32, 10, 50, 7, 45, -1),      # partial fill: x edges at bytes 21 and 135 cut 16-byte chunks
    (20, 32, 60, 96, 70, 96, -1),    # touches the bottom / right crop edges and the last frame
    (5, 20, 0, 31, 81, 96, 2),       # copy from another frame, top / right edges
    (10, 20, 30, 70, 29, 67, 15),    # src inside its own box
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


def _occlude(win, box, fill):
    """numpy statement of the box rule on one uint8 window (T, H, W, 3)."""
    t0, t1, y0, y1, x0, x1, src = box
    out = win.copy()
    if t0 < t1 and y0 < y1 and x0 < x1:
        out[t0:t1, y0:y1, x0:x1] = fill if src < 0 else win[src, y0:y1, x0:x1][None]
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
                                 (C.c_int32 * n)(*starts), (C.c_int32 * n)(*[int(x) for x in a_starts]), n, p.chunk_size, mel.data_ptr(),
                                 int(mel.shape[1]), int(mel.shape[2]), total_v_frames, chunk_a_size, prec, batch, out.data_ptr(), ws.data_ptr(),
                                 ws.numel(), torch.cuda.current_stream().cuda_stream)
        _cabi.check(h.ptr, rc)
    return out.cpu()


def _host_reference(p, track, starts, mel, total_v_frames, boxes, fill, chunk_a_size=128):
    """(n, K) logits: every (window, box) occluded with numpy, the occluded windows laid end to end as one track and scored by
    lsd_score_windows with the window's own audio start."""
    T = p.chunk_size
    host = track.cpu().numpy()
    wins = [_occlude(host[s:s + T], b, fill) for s in starts for b in boxes]
    flat = torch.from_numpy(np.concatenate(wins)).cuda()
    a = [p._audio_start(s, int(mel.shape[2]), total_v_frames, chunk_a_size) for s in starts for _ in boxes]
    ref = _score_windows_explicit(p, flat, [r * T for r in range(len(wins))], mel, total_v_frames, a, chunk_a_size)
    return ref.view(len(starts), len(boxes))


def _track(seed, n_frames=200, H=96, W=96, Ta_full=800):
    g = torch.Generator().manual_seed(seed)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    mel = (-80.0 * torch.rand((1, 80, Ta_full), generator=g)).cuda()
    return track, mel


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_occlusions_bitwise(model, prec):
    """Every (window, box) logit equals the plain forward of the host-occluded window; the empty box equals score_track_logits."""
    model.compute_precision = prec
    track, mel = _track(51)
    n_frames = 200
    starts = list(range(0, n_frames - 32 + 1, 21))                   # 9 windows: 63 rows, 4 batches of 16 (pipelined on bf16)
    p = lb.Predictor(model, batch_size=16)
    out = p.score_track_occlusions(track, starts, mel, n_frames, BOXES, fill=37).cpu()
    assert out.shape == (len(starts), len(BOXES)) and out.dtype == torch.float32
    ref = _host_reference(p, track, starts, mel, n_frames, BOXES, 37)
    for k in range(len(BOXES)):
        assert torch.equal(out[:, k], ref[:, k]), (k, out[:, k], ref[:, k])
    assert torch.equal(out[:, 0], p.score_track_logits(track, starts, mel, n_frames).cpu())
    assert not torch.equal(out[:, 3], out[:, 0])                      # the occlusion changed something


def _occlusions_raw(model, track, starts, mel, n_frames, boxes, fill, batch, ws_bytes, T=32, Ta=128):
    """lsd_score_occlusions straight through the C-ABI, in a workspace of exactly ws_bytes (called twice: the second call reuses
    the zero padding of the first)."""
    L = _cabi.lib()
    n, K = len(starts), len(boxes)
    H, W = int(track.shape[1]), int(track.shape[2])
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        L.lsd_workspace_invalidate(h.ptr)
        logits = torch.empty(n, K, dtype=torch.float32, device="cuda")
        bc = (_cabi.LsdOcclusion * K)(*[_cabi.LsdOcclusion(*b) for b in boxes])
        for _ in range(2):
            rc = L.lsd_score_occlusions(h.ptr, track.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*starts), None, n, T, mel.data_ptr(),
                                        int(mel.shape[1]), int(mel.shape[2]), n_frames, Ta, bc, K, fill, model._precision(), batch,
                                        logits.data_ptr(), ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
            _cabi.check(h.ptr, rc)
            out = logits.cpu()
        L.lsd_workspace_invalidate(h.ptr)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("misaligned", [False, True])
def test_occlusions_batches_and_exact_workspace(model, misaligned):
    """batch=7 over 54 rows (7 full batches and a short one of 5): pipelined in a double workspace and again in exactly the queried
    workspace, both equal to one batch of 64.  misaligned: a track that is not 16-byte aligned takes the byte-wise occlusion route."""
    model.compute_precision = "bf16"
    n_frames, H, W = 200, 96, 96
    g = torch.Generator().manual_seed(52)
    data = torch.randint(0, 256, (n_frames * H * W * 3 + 16,), generator=g, dtype=torch.uint8).cuda()
    o = 1 if misaligned else 0
    track = data[o:o + n_frames * H * W * 3].view(n_frames, H, W, 3)
    mel = (-80.0 * torch.rand((1, 80, 800), generator=g)).cuda()
    starts = list(range(0, 169, 21))                                  # 9 windows
    boxes = BOXES[1:]                                                 # K = 6
    L = _cabi.lib()
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        need7 = L.lsd_score_occlusions_workspace_bytes(h.ptr, 7, 32, H, W, 80, 128, _cabi.LSD_PREC_BF16)
        need64 = L.lsd_score_occlusions_workspace_bytes(h.ptr, 64, 32, H, W, 80, 128, _cabi.LSD_PREC_BF16)
    assert 0 < need7 < need64
    one = _occlusions_raw(model, track, starts, mel, n_frames, boxes, 128, 64, need64)
    piped = _occlusions_raw(model, track, starts, mel, n_frames, boxes, 128, 7, 2 * need7)
    exact = _occlusions_raw(model, track, starts, mel, n_frames, boxes, 128, 7, need7)
    assert torch.equal(piped, one) and torch.equal(exact, one)
    if misaligned:
        p = lb.Predictor(model, batch_size=64)
        assert torch.equal(one, _host_reference(p, track.contiguous(), starts, mel, n_frames, boxes, 128))


@pytest.mark.gpu
def test_occlusions_second_geometry(model):
    """T=16 windows of 64x64 crops, 64 mel columns, bf16."""
    model.compute_precision = "bf16"
    track, mel = _track(53, n_frames=120, H=64, W=64, Ta_full=480)
    n_frames = 120
    starts = [0, 9, 40, 77, 104]
    p = lb.Predictor(model, chunk_size=16, batch_size=8)
    boxes = [(0, 0, 0, 0, 0, 0, -1), (4, 8, 0, 64, 0, 64, 3), (0, 4, 0, 64, 0, 64, 4), (0, 16, 5, 37, 11, 43, -1),
             (12, 16, 40, 64, 50, 64, 13)] + p.fill_cell_boxes(16, 64, 64, 2)
    out = p.score_track_occlusions(track, starts, mel, n_frames, boxes, fill=200, chunk_a_size=64).cpu()
    ref = _host_reference(p, track, starts, mel, n_frames, boxes, 200, chunk_a_size=64)
    assert torch.equal(out, ref)


@pytest.mark.gpu
def test_occlusion_argument_errors(model):
    """Bad arguments raise ValueError (LSD_ERR_SHAPE / LSD_ERR_ARG at the C-ABI) before anything is launched."""
    model.compute_precision = "bf16"
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8, device="cuda")
    mel = torch.zeros((1, 80, 300), device="cuda")
    p = lb.Predictor(model, batch_size=4)
    good = [(0, 0, 0, 0, 0, 0, -1)]
    bad_boxes = [[], [good[0]] * 1025, [(0, 33, 0, 96, 0, 96, -1)], [(-1, 4, 0, 96, 0, 96, -1)], [(4, 3, 0, 96, 0, 96, -1)],
                 [(0, 4, 10, 9, 0, 96, -1)], [(0, 4, 0, 97, 0, 96, -1)], [(0, 4, 0, 96, 5, 97, -1)], [(0, 4, 0, 96, 0, 96, 32)],
                 [(0, 4, 0, 96, 0, 96, -2)], [(0, 4, 0, 96, 0, 96)]]
    n0 = model.launch_count()
    for b in bad_boxes:
        with pytest.raises(ValueError):
            p.score_track_occlusions(track, [0, 8], mel, 64, b)
    with pytest.raises(ValueError):
        p.score_track_occlusions(track, [0, 40], mel, 64, good)          # window [40, 72) outside the 64-frame track
    with pytest.raises(ValueError):
        p.score_track_occlusions(track, [0], mel, 64, good, fill=256)
    # the C-ABI itself
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    ws = model._workspace(1 << 20, track.device)
    out = torch.empty(2, 2, device="cuda")
    st = (C.c_int32 * 2)(0, 8)

    def call(boxes, K, fill=128, starts=st):
        return L.lsd_score_occlusions(h.ptr, track.data_ptr(), 64, 96, 96, starts, None, 2, 32, mel.data_ptr(), 80, 300, 64, 128,
                                      boxes, K, fill, _cabi.LSD_PREC_BF16, 2, out.data_ptr(), ws.data_ptr(), ws.numel(), None)

    one = (_cabi.LsdOcclusion * 1)(_cabi.LsdOcclusion(0, 0, 0, 0, 0, 0, -1))
    assert call(None, 1) == _cabi.LSD_ERR_ARG
    assert call(one, 0) == _cabi.LSD_ERR_SHAPE
    assert call(one, 1, fill=-1) == _cabi.LSD_ERR_ARG
    assert call((_cabi.LsdOcclusion * 1)(_cabi.LsdOcclusion(0, 4, 0, 96, 0, 96, 40)), 1) == _cabi.LSD_ERR_SHAPE
    assert call((_cabi.LsdOcclusion * 1)(_cabi.LsdOcclusion(0, 4, 0, 96, 90, 80, -1)), 1) == _cabi.LSD_ERR_SHAPE
    assert call(one, 1, starts=(C.c_int32 * 2)(0, 33)) == _cabi.LSD_ERR_SHAPE
    assert model.launch_count() == n0


@pytest.mark.gpu
def test_explain_track_matches_its_logits(model):
    model.compute_precision = "bf16"
    track, mel = _track(54)
    n_frames = 200
    starts = list(range(0, 169, 24))                                   # 8 windows
    p = lb.Predictor(model, batch_size=64)
    ex = p.explain_track(track, starts, mel, n_frames)
    T, S, g = 32, 8, 4
    boxes = [(0, 0, 0, 0, 0, 0, -1)] + p.freeze_segment_boxes(T, 4) + p.fill_cell_boxes(T, 96, 96, 4)
    logits = p.score_track_occlusions(track, starts, mel, n_frames, boxes).cpu().numpy()
    probs = np.array([[p._calibrate(float(x)) for x in row] for row in logits])
    assert np.array_equal(ex["confidence"], probs[:, 0])
    assert np.array_equal(ex["temporal"], probs[:, 1:1 + S] - probs[:, :1])
    assert np.array_equal(ex["spatial"], (probs[:, 1 + S:] - probs[:, :1]).reshape(len(starts), g, g))
    assert np.allclose(ex["spatial_mean"], ex["spatial"].mean(axis=0))
    first, tl = frame_evidence_timeline(starts, ex["temporal"], 4, T)
    assert ex["frame_first"] == first == 0 and ex["frame_evidence"] == tl and len(tl) == starts[-1] + T
    assert (ex["segment_frames"], ex["grid"], ex["fill"]) == (4, 4, 128)
    # the confidence column is the plain window score
    plain = [p._calibrate(float(x)) for x in p.score_track_logits(track, starts, mel, n_frames).cpu().tolist()]
    assert ex["confidence"].tolist() == plain


@pytest.mark.gpu
def test_long_video_evidence_entry_on_gpu(model):
    """evidence=True: `confidence` equals the selected track's window confidences, every other result key is unchanged."""
    model.compute_precision = "bf16"
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(model, batch_size=16)
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, evidence=True)
    assert set(res) == set(base) | {"evidence"}
    ev = res["evidence"]
    sel = next(t for t in res["tracks"] if t["track_id"] == res["selected_track_id"])
    assert ev["track_id"] == res["selected_track_id"]
    assert ev["confidence"].tolist() == sel["window_confidences"]
    tr = next(t for t in tracks if int(t["track_id"]) == ev["track_id"])
    assert ev["frame_first"] == min(int(s) for s in tr["chunk_starts"])   # absolute video frames
    for k in base:
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_freeze_segment_boxes():
    P = lb.Predictor
    b = P.freeze_segment_boxes(32, 4)
    assert len(b) == 8 and b[0] == (0, 4, 0, 96, 0, 96, 4) and b[1] == (4, 8, 0, 96, 0, 96, 3) and b[7] == (28, 32, 0, 96, 0, 96, 27)
    assert P.freeze_segment_boxes(10, 4, 64, 48) == [(0, 4, 0, 64, 0, 48, 4), (4, 8, 0, 64, 0, 48, 3), (8, 10, 0, 64, 0, 48, 7)]
    assert P.freeze_segment_boxes(2, 1) == [(0, 1, 0, 96, 0, 96, 1), (1, 2, 0, 96, 0, 96, 0)]
    for s in (0, 32, 40):
        with pytest.raises(ValueError):
            P.freeze_segment_boxes(32, s)


def test_fill_cell_boxes():
    P = lb.Predictor
    b = P.fill_cell_boxes(32, 96, 96, 4)
    assert len(b) == 16 and b[0] == (0, 32, 0, 24, 0, 24, -1) and b[1] == (0, 32, 0, 24, 24, 48, -1) and b[15] == (0, 32, 72, 96, 72, 96, -1)
    b = P.fill_cell_boxes(16, 10, 20, 3)                                # edges round(j*10/3) = 0, 3, 7, 10 and 0, 7, 13, 20
    assert [(y0, y1) for _, _, y0, y1, _, _, _ in b[::3]] == [(0, 3), (3, 7), (7, 10)]
    assert [(x0, x1) for _, _, _, _, x0, x1, _ in b[:3]] == [(0, 7), (7, 13), (13, 20)]
    for g in (0, 11):
        with pytest.raises(ValueError):
            P.fill_cell_boxes(16, 10, 20, g)


def test_frame_evidence_timeline_hand_computed():
    # windows at 10 and 14, T = 8, segments of 4: frames 10-13 only window 0 (0.1), 14-17 both (0.3 and 0.5), 18-21 window 1
    first, v = frame_evidence_timeline([10, 14], [[0.1, 0.3], [0.5, -0.2]], 4, 8)
    assert first == 10 and len(v) == 12
    assert v[:4] == pytest.approx([0.1] * 4) and v[4:8] == pytest.approx([0.4] * 4) and v[8:] == pytest.approx([-0.2] * 4)
    # uneven last segment (T = 8, segments of 3: [0,3), [3,6), [6,8)) and a gap no window covers
    first, v = frame_evidence_timeline([0, 12], [[1, 2, 3], [4, 5, 6]], 3, 8)
    assert first == 0 and v == [1, 1, 1, 2, 2, 2, 3, 3, None, None, None, None, 4, 4, 4, 5, 5, 5, 6, 6]
    assert frame_evidence_timeline([], np.zeros((0, 2)), 4, 8) == (0, [])
    with pytest.raises(ValueError):
        frame_evidence_timeline([0], [[0.1, 0.2, 0.3]], 4, 8)


def test_long_video_evidence_entry():
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def evidence_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"confidence": np.full(len(tr["chunk_starts"]), 0.7), "frame_first": int(tr["chunk_starts"][0])}

    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, evidence=True, evidence_fn=evidence_fn, **fns)
    assert "evidence" not in base
    assert set(res) == set(base) | {"evidence"}
    assert res["evidence"]["track_id"] == res["selected_track_id"] == seen[0] and len(seen) == 1
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k
