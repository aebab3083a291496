"""Audio-visual offset sweep: `LipSyncModel.forward_audio_variants` (lsd_forward_audio_variants), `Predictor.score_track_offsets`
(lsd_score_offsets), `aggregate.av_offset_profile` and the `av_offset` entry of `predict_long_video_from_tracks`.
The logit of (window, offset) must be bit for bit the plain forward's logit for that window with that audio slice."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import av_offset_profile
from oracle import lipsync_oracle as orc
from tests.golden.long_video_synth import SCENARIOS, make_audio, make_tracks


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()


@pytest.fixture(scope="module")
def model(built, seed0_sd):
    m = lb.LipSyncModel()
    m.load_state_dict(seed0_sd, strict=True)
    return m.to("cuda:0").eval()


def _variants(seed, B, K, t=32, ta=128):
    video, _ = lb.synthetic_windows(seed, B, t=t, ta=ta)
    _, audio = lb.synthetic_windows(seed + 100, B * K, t=1, ta=ta)
    return video.cuda(), audio.view(B, K, *audio.shape[1:]).cuda()


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("B,K,t,ta,rows", [(3, 4, 32, 128, None), (3, 3, 16, 64, None), (21, 5, 32, 128, "32")])
def test_tensor_variants_bitwise(model, monkeypatch, prec, B, K, t, ta, rows):
    """forward_audio_variants(v, a)[:, k] == model(v, a[:, k]) bit for bit; rows="32" splits B*K = 105 rows into audio
    groups of 6 videos (several groups, a shorter last one)."""
    if rows:
        monkeypatch.setenv("LSD_VARIANT_ROWS", rows)
    model.compute_precision = prec
    v, a = _variants(7, B, K, t, ta)
    out = model.forward_audio_variants(v, a).cpu()
    assert out.shape == (B, K) and out.dtype == torch.float32
    for k in range(K):
        ref = model(v, a[:, k].contiguous()).cpu()
        assert torch.equal(out[:, k], ref), (k, out[:, k], ref)


@pytest.mark.gpu
def test_tensor_variants_fallback_route_bitwise(model, monkeypatch):
    """The launch-by-launch token path (LSD_TOK_FRONT=0) scores one plain forward per variant: same bits as forward()."""
    monkeypatch.setenv("LSD_TOK_FRONT", "0")
    model.compute_precision = "bf16"
    v, a = _variants(8, 2, 3)
    out = model.forward_audio_variants(v, a).cpu()
    for k in range(3):
        assert torch.equal(out[:, k], model(v, a[:, k].contiguous()).cpu())


def _score_windows_explicit(p, track, starts, mel, n_frames, a_starts, chunk_a_size=128):
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
                                 int(mel.shape[1]), int(mel.shape[2]), n_frames, chunk_a_size, prec, batch, out.data_ptr(), ws.data_ptr(),
                                 ws.numel(), torch.cuda.current_stream().cuda_stream)
        _cabi.check(h.ptr, rc)
    return out.cpu()


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_track_offsets_bitwise_and_effective_starts(model, prec):
    model.compute_precision = prec
    g = torch.Generator().manual_seed(41)
    n_frames = 200
    track = torch.randint(0, 256, (n_frames, 96, 96, 3), generator=g, dtype=torch.uint8).cuda()
    mel = (-80.0 * torch.rand((1, 80, 800), generator=g)).cuda()
    starts = list(range(0, n_frames - 32 + 1, 8))                    # 22 windows
    offsets = [-40, -7, 0, 3, 7, 40]
    p = lb.Predictor(model, batch_size=8)                             # 3 batches (pipelined in lsd_score_windows on bf16)
    logits, eff, valid = p.score_track_offsets(track, starts, mel, n_frames, offsets)
    logits = logits.cpu()
    assert logits.shape == (len(starts), len(offsets)) and eff.dtype == np.int32 and valid.dtype == bool
    # effective starts / valid: _audio_start(v) + d under the clamp rule
    Ta_full, Ta = 800, 128
    base = np.array([p._audio_start(s, Ta_full, n_frames, Ta) for s in starts])[:, None]
    moved = base + np.array(offsets)[None, :]
    assert np.array_equal(eff, np.maximum(np.minimum(moved, Ta_full - Ta), 0))
    assert np.array_equal(valid, (moved >= 0) & (moved <= Ta_full - Ta))
    assert valid.any() and not valid.all()                            # both clip ends clamp
    for k in range(len(offsets)):
        ref = _score_windows_explicit(p, track, starts, mel, n_frames, eff[:, k])
        assert torch.equal(logits[:, k], ref), k
    assert torch.equal(logits[:, offsets.index(0)], p.score_track_logits(track, starts, mel, n_frames).cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("misaligned", [False, True])
def test_track_offsets_short_last_batch_exact_workspace(model, monkeypatch, misaligned):
    """The group size of every batch follows `batch`, so the last, shorter batch fits the workspace lsd_score_offsets_workspace_bytes
    reports for `batch`: 32 rows per group and K = 6 give groups of 4 videos; 12 windows in batches of 7 end with a batch of 5
    (groups 4 + 1).  misaligned: a track that is not 16-byte aligned takes the gather route instead of reading it in place."""
    monkeypatch.setenv("LSD_VARIANT_ROWS", "32")
    model.compute_precision = "bf16"
    g = torch.Generator().manual_seed(43)
    n_frames, H, W, T, Ta, K, batch = 120, 32, 32, 32, 128, 6, 7
    data = torch.randint(0, 256, (n_frames * H * W * 3 + 16,), generator=g, dtype=torch.uint8).cuda()
    o = 1 if misaligned else 0
    track = data[o:o + n_frames * H * W * 3].view(n_frames, H, W, 3)
    mel = (-80.0 * torch.rand((1, 80, 480), generator=g)).cuda()
    starts = [8 * i for i in range(12)]
    offsets = [-9, -3, 0, 2, 5, 11]
    L = _cabi.lib()
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        need = L.lsd_score_offsets_workspace_bytes(h.ptr, batch, K, T, H, W, 80, Ta, _cabi.LSD_PREC_BF16)
        assert need > 0
        ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        L.lsd_workspace_invalidate(h.ptr)
        logits = torch.empty(len(starts), K, dtype=torch.float32, device="cuda")
        eff_c = (C.c_int32 * (len(starts) * K))()
        for _ in range(2):                                            # the second call reuses the zero padding of the first
            rc = L.lsd_score_offsets(h.ptr, track.data_ptr(), n_frames, H, W, (C.c_int32 * 12)(*starts), None, 12, T, mel.data_ptr(), 80,
                                     480, n_frames, Ta, (C.c_int32 * K)(*offsets), K, _cabi.LSD_PREC_BF16, batch, logits.data_ptr(), eff_c,
                                     ws.data_ptr(), need, torch.cuda.current_stream().cuda_stream)
            _cabi.check(h.ptr, rc)
            out = logits.cpu()
        L.lsd_workspace_invalidate(h.ptr)
    eff = np.frombuffer(eff_c, dtype=np.int32).reshape(12, K)
    p = lb.Predictor(model, batch_size=batch)
    for k in range(K):
        assert torch.equal(out[:, k], _score_windows_explicit(p, track, starts, mel, n_frames, eff[:, k])), k


@pytest.mark.gpu
def test_visual_side_runs_once(model):
    """Launches per call do not depend on K on the shared route (with the bitwise test: the visual encoder runs once)."""
    model.compute_precision = "bf16"
    counts = {}
    for K in (1, 8):
        v, a = _variants(9, 3, K)
        model.forward_audio_variants(v, a)                            # warm-up: stage programs of these shapes
        n0 = model.launch_count()
        model.forward_audio_variants(v, a)
        counts[K] = model.launch_count() - n0
    assert counts[1] == counts[8] > 0, counts


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_variants_against_oracle(model, seed0_sd, prec):
    model.compute_precision = prec
    v, a = _variants(10, 2, 3)
    out = model.forward_audio_variants(v, a).cpu()
    for k in range(3):
        ref = orc.forward(seed0_sd, v.cpu(), a[:, k].cpu())
        if prec == "fp32":
            assert float((out[:, k] - ref).abs().max()) / float(ref.abs().max()) <= 1e-4
        else:
            assert float((out[:, k] - ref).abs().max()) <= 2e-2
        assert ((out[:, k] >= 0) == (ref >= 0)).all()


@pytest.mark.gpu
def test_variant_errors(model):
    model.compute_precision = "bf16"
    v, a = _variants(11, 2, 2)
    with pytest.raises(ValueError):
        model.forward_audio_variants(v, a[:, :0])                     # K = 0
    with pytest.raises(ValueError):
        model.forward_audio_variants(v, a[:, :1].expand(2, 65, 1, 80, 128).contiguous())
    with pytest.raises(ValueError):
        model.forward_audio_variants(v, a[:, 0])                      # (B,1,F,Ta): rank 4
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8, device="cuda")
    mel = torch.zeros((1, 80, 300), device="cuda")
    p = lb.Predictor(model, batch_size=4)
    for offs in ([], list(range(65))):
        with pytest.raises(ValueError):
            p.score_track_offsets(track, [0, 8], mel, 64, offs)
    # the C-ABI itself: K out of range -> LSD_ERR_SHAPE, no offsets -> LSD_ERR_ARG
    L = _cabi.lib()
    h = model._lsd_handle
    ws = model._workspace(1 << 20, v.device)
    st = (C.c_int32 * 2)(0, 8)
    args = (h.ptr, track.data_ptr(), 64, 96, 96, st, None, 2, 32, mel.data_ptr(), 80, 300, 64, 128)
    tail = (_cabi.LSD_PREC_BF16, 2, ws.data_ptr(), None, ws.data_ptr(), ws.numel(), None)
    assert L.lsd_score_offsets(*args, None, 1, *tail) == _cabi.LSD_ERR_ARG
    assert L.lsd_score_offsets(*args, (C.c_int32 * 1)(0), 0, *tail) == _cabi.LSD_ERR_SHAPE
    assert L.lsd_forward_audio_variants(h.ptr, v.data_ptr(), _cabi.LSD_F32, _cabi.LSD_NCDHW, a.data_ptr(), _cabi.LSD_F32, 2, 0, 32, 96, 96,
                                        80, 128, _cabi.LSD_PREC_BF16, ws.data_ptr(), ws.data_ptr(), ws.numel(), None) == _cabi.LSD_ERR_SHAPE


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_profile_argmax_invalid_and_empty():
    confs = np.array([[0.9, 0.2, 0.6, 0.1], [0.9, 0.4, 0.8, 0.3], [0.9, 0.6, 0.7, 0.2]], np.float32)
    valid = np.ones_like(confs, bool)
    valid[:, 0] = False                                               # offset -3: no valid window
    valid[2, 2] = False
    r = av_offset_profile(confs, valid, [-3, 0, 2, 5], "median", 0.1)
    assert r["profile"][0] is None and r["n_valid"] == [0, 3, 2, 3]
    assert r["profile"][1] == pytest.approx(0.4) and r["profile"][2] == pytest.approx(0.7) and r["profile"][3] == pytest.approx(0.2)
    assert r["best_offset"] == 2 and r["best_confidence"] == pytest.approx(0.7)
    assert r["confidence_at_zero"] == pytest.approx(0.4) and r["margin"] == pytest.approx(0.3)
    r = av_offset_profile(confs, np.zeros_like(valid), [-3, 0, 2, 5])
    assert r["best_offset"] is None and r["margin"] is None and r["profile"] == [None] * 4


def test_profile_tie_break():
    c = np.full((2, 5), 0.5, np.float32)
    v = np.ones((2, 5), bool)
    assert av_offset_profile(c, v, [-4, -2, 2, 4, 7])["best_offset"] == -2     # smaller |d|, then smaller d
    assert av_offset_profile(c[:, :4], v[:, :4], [3, -1, 0, 1])["best_offset"] == 0
    assert av_offset_profile(c[:, :2], v[:, :2], [6, 3])["best_offset"] == 3
    r = av_offset_profile(c[:, :2], v[:, :2], [6, 3])
    assert r["confidence_at_zero"] is None and r["margin"] is None


@pytest.mark.parametrize("smoothing,expect", [("median", 0.3), ("none", 0.4), ("trimmed_mean", 0.3)])
def test_profile_robust_method(smoothing, expect):
    col = np.array([0.1, 0.2, 0.3, 0.4, 1.0], np.float32)[:, None]
    r = av_offset_profile(col, np.ones_like(col, bool), [0], smoothing, 0.2)
    assert r["profile"][0] == pytest.approx(expect)


def test_long_video_av_offset_entry():
    spec_name = sorted(SCENARIOS)[0]
    spec = SCENARIOS[spec_name]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def offset_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"best_offset": 4, "offsets": [0, 4]}

    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, av_offset=True, offset_fn=offset_fn, **fns)
    assert "av_offset" not in base
    assert set(res) == set(base) | {"av_offset"}
    assert res["av_offset"]["best_offset"] == 4 and res["av_offset"]["track_id"] == res["selected_track_id"] == seen[0]
    assert len(seen) == 1
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k
