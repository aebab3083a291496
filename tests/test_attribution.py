"""Branch attribution: `Predictor.score_track_branch_features` (lsd_score_branch_features), `Predictor.branch_attribution`
(lsd_branch_attribution), `Predictor.attribution_track`, `aggregate.branch_attribution_summary` and the `attribution` entry of
`predict_long_video_from_tracks`.  oracle/attribution_oracle.py restates the head, the hybrid rows, the coalition values and the
Shapley values in float64."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import branch_attribution_summary, frame_evidence_timeline
from lipsync_b200.long_video import _track_u8
from oracle import attribution_oracle as ato
from oracle import lipsync_oracle as orc
from tests.golden.long_video_synth import SCENARIOS, make_audio, make_tracks

P = lb.Predictor
SL = ato.SLICES


# ---------------------------------------------------------------------------------------------------------------- CPU
def _game(fn):
    """(1, 16) coalition values of the set function fn(frozenset of players)."""
    return np.array([[fn(frozenset(p for p in range(4) if (S >> p) & 1)) for S in range(16)]], dtype=np.float64)


def test_shapley_hand_games():
    # additive game: every player gets its own worth
    phi = ato.shapley(_game(lambda s: sum((1.0, 2.0, -3.0, 0.5)[p] for p in s)))
    assert np.allclose(phi, [[1.0, 2.0, -3.0, 0.5]], atol=1e-15)
    # unanimity game of {0, 1}: the worth 6 is split evenly, players 2 and 3 are dummies
    phi = ato.shapley(_game(lambda s: 6.0 if {0, 1} <= s else 0.0))
    assert np.allclose(phi, [[3.0, 3.0, 0.0, 0.0]], atol=1e-15)
    # majority game (any 3 of 4): symmetric, 1/4 each
    phi = ato.shapley(_game(lambda s: 1.0 if len(s) >= 3 else 0.0))
    assert np.allclose(phi, [[0.25] * 4], atol=1e-15)
    # player 0 alone is worth 4, with player 1 the pair is worth 10: phi = (4 + 3, 3, 0, 0), p3 a dummy, sums to v(15) - v(0)
    v = _game(lambda s: (4.0 if 0 in s else 0.0) + (6.0 if {0, 1} <= s else 0.0) + 1.0)
    phi = ato.shapley(v)
    assert np.allclose(phi, [[7.0, 3.0, 0.0, 0.0]], atol=1e-14)
    assert np.isclose(phi.sum(), v[0, 15] - v[0, 0])
    # random game in which players 1 and 2 are interchangeable and player 3 is a dummy: efficiency, symmetry, dummy gets 0
    base = np.random.default_rng(0).normal(size=6)
    v = _game(lambda s: base[(0 in s) + 2 * len({1, 2} & s)])
    phi = ato.shapley(v)
    assert np.isclose(phi.sum(), v[0, 15] - v[0, 0], atol=1e-12)
    assert abs(phi[0, 1] - phi[0, 2]) < 1e-12 and abs(phi[0, 3]) < 1e-12


def test_oracle_head_is_the_reference_head(seed0_sd):
    """With the background equal to the window, every coalition value is f(x) = classifier(cat[cls, artifact_fusion(x)])."""
    g = np.random.default_rng(1)
    x = g.normal(size=(5, 448)) * np.r_[np.full(256, 1.0), np.abs(g.normal(size=192))]
    sd = {k: v.double() for k, v in seed0_sd.items() if v.is_floating_point()}
    xt = torch.from_numpy(x)
    p = "artifact_detector.artifact_fusion"
    art = torch.relu(torch.relu(xt @ sd[p + ".0.weight"].t() + sd[p + ".0.bias"]) @ sd[p + ".2.weight"].t() + sd[p + ".2.bias"])
    ref = orc.classifier(sd, torch.cat([xt[:, :256], art], dim=-1)).numpy()
    assert np.allclose(ato.head(seed0_sd, x), ref, rtol=0, atol=1e-12)
    for i in range(5):
        v = ato.coalition_values(seed0_sd, x[i:i + 1], x[i:i + 1])
        assert np.allclose(v, ref[i], rtol=0, atol=1e-12)
    # hybrid rows take slice p from the window exactly when bit p is set
    a, b = np.zeros((1, 448)), np.ones((1, 448))
    for S in range(16):
        h = ato.hybrid(a, b, S)
        for p, (lo, hi) in enumerate(SL):
            assert (h[0, lo:hi] == (0.0 if (S >> p) & 1 else 1.0)).all()


def test_summary_hand_built():
    phi = np.array([[-2.0, 0.5, 0.1, 0.0],      # fake window: sync most negative
                    [0.2, -0.1, 3.0, 0.4],      # real window: delta most positive
                    [-0.3, -0.2, 0.0, -1.0],    # fake window: hf most negative
                    [1.0, 0.0, 0.0, 0.2]])      # real window: sync most positive
    probs = np.array([0.1, 0.9, 0.3, 0.6])
    res = branch_attribution_summary(phi, probs, 0.5, "median", 0.1, starts=[0, 8, 16, 60], T=32)
    assert np.allclose(res["mean_phi"], phi.mean(axis=0)) and np.allclose(res["median_phi"], np.median(phi, axis=0))
    mag = np.abs(phi).mean(axis=0)
    assert np.allclose(res["share"], mag / mag.sum()) and np.isclose(res["share"].sum(), 1.0)
    assert res["leading_branch"] == ["sync", "delta", "hf", "sync"]
    # median of (0.1, 0.9, 0.3, 0.6) = 0.45: fake; mean phi = (-0.275, 0.05, 0.775, -0.1): sync pushes hardest toward fake
    assert res["verdict"] == "fake" and np.isclose(res["confidence"], 0.45) and res["verdict_driver"] == "sync"
    res_real = branch_attribution_summary(phi, probs, 0.4, "median", 0.1)
    assert res_real["verdict"] == "real" and res_real["verdict_driver"] == "delta" and "frame_timeline" not in res_real
    assert res_real["leading_branch"] == ["sync", "delta", "hf", "sync"]
    # timeline: frame f holds the mean phi of the windows covering it; frames 48..59 are covered by no window
    assert res["frame_first"] == 0 and set(res["frame_timeline"]) == set(ato.BRANCHES)
    sync = res["frame_timeline"]["sync"]
    assert len(sync) == 92 and sync[0] == -2.0 and np.isclose(sync[10], -0.9) and np.isclose(sync[20], -0.7)
    assert sync[50] is None and sync[91] == 1.0
    for b, name in enumerate(ato.BRANCHES):
        assert res["frame_timeline"][name] == frame_evidence_timeline([0, 8, 16, 60], phi[:, b:b + 1], 32, 32)[1]
    # all-zero attributions: zero shares
    z = branch_attribution_summary(np.zeros((2, 4)), [0.7, 0.8])
    assert (z["share"] == 0).all() and z["verdict"] == "real"
    with pytest.raises(ValueError):
        branch_attribution_summary(np.zeros((2, 3)), [0.5, 0.5])
    with pytest.raises(ValueError):
        branch_attribution_summary(np.zeros((2, 4)), [0.5])
    with pytest.raises(ValueError):
        branch_attribution_summary(np.zeros((2, 4)), [0.5, 0.5], starts=[0])


def test_track_background_index():
    assert P.track_background_index(1) == [0]
    assert P.track_background_index(5) == [0, 1, 2, 3, 4]
    assert P.track_background_index(64) == list(range(64))
    idx = P.track_background_index(300)
    assert len(idx) == 64 and idx == [(k * 300) // 64 for k in range(64)] and idx[-1] == 295
    assert P.track_background_index(1600)[:3] == [0, 25, 50]


def test_branch_attribution_value_errors():
    pred = lb.Predictor(None, device=torch.device("cpu"))
    f = torch.zeros(3, 448)
    for feats, bg in [(torch.zeros(3, 447), f[:1]), (f, torch.zeros(2, 448, 1)), (f.double(), f[:1]), (f, f[:1].half()),
                      (f, torch.zeros(0, 448)), (f, torch.zeros(257, 448)), (f, torch.zeros(1, 448, device="meta")),
                      (torch.zeros(3, 448, device="meta"), f[:1]), (f.numpy(), f[:1]), (f, f[:1])]:
        with pytest.raises(ValueError):
            pred.branch_attribution(feats, bg)            # the last pair is valid but the predictor has no CUDA model
    with pytest.raises(ValueError):
        pred.attribution_track(torch.zeros(40, 96, 96, 3, dtype=torch.uint8), [0], torch.zeros(1, 80, 200), 40, background="window")


def test_long_video_attribution_entry():
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def attribution_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"verdict_driver": "hf", "background": "track", "window_starts": [int(s) for s in tr["chunk_starts"]]}

    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, attribution=True,
                                            attribution_fn=attribution_fn, **fns)
    assert "attribution" not in base
    assert set(res) == set(base) | {"attribution"}
    assert res["attribution"]["track_id"] == res["selected_track_id"] == seen[0] and len(seen) == 1
    assert res["attribution"]["verdict_driver"] == "hf"
    tr = next(t for t in tracks if int(t["track_id"]) == seen[0])
    assert res["attribution"]["window_starts"] == [int(s) for s in tr["chunk_starts"]]
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k


def test_long_video_attribution_default_hook(monkeypatch):
    """The default hook calls attribution_track on the selected track with its absolute window starts, the call's threshold and
    the given background (the track's own windows when None)."""
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    calls = []

    def fake(track, starts, mel_full, total_v, background="track", confidence_threshold=0.5, audio_starts_from=None):
        calls.append((background, confidence_threshold, list(audio_starts_from)))
        return {"window_starts": list(audio_starts_from)}

    monkeypatch.setattr(pred, "attribution_track", fake)
    fns = dict(score_fn=lambda t: [0.7] * len(t["chunk_starts"]), speech_fn=lambda t, idxs: [0.6] * len(idxs),
               mouth_fn=lambda t: {"check_result": "no_data"})
    ref_bg = torch.zeros(3, 448)
    for bg, want in [(None, "track"), (ref_bg, ref_bg)]:
        res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, attribution=True,
                                                attribution_background=bg, confidence_threshold=0.4, **fns)
        tr = next(t for t in tracks if int(t["track_id"]) == res["selected_track_id"])
        assert calls[-1][0] is want and calls[-1][1] == 0.4 and calls[-1][2] == [int(s) for s in tr["chunk_starts"]]


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


N_FRAMES, TA_FULL = 400, 1600


def _track(seed, n_frames=N_FRAMES, Ta_full=TA_FULL):
    g = torch.Generator().manual_seed(seed)
    track = torch.randint(0, 256, (n_frames, 96, 96, 3), generator=g, dtype=torch.uint8)
    track[::4, :40, :30] = 255
    mel = (-80.0 * torch.rand((1, 80, Ta_full), generator=g)).cuda()
    return track.cuda(), mel


def _starts(n):
    return [(i * 7) % (N_FRAMES - 32 + 1) for i in range(n)]


@pytest.fixture(scope="module")
def feats300(model):
    """Exported head inputs of 300 windows (bf16 route) and 64 more as a background source."""
    model.compute_precision = "bf16"
    track, mel = _track(5)
    p = lb.Predictor(model)
    _, f = p.score_track_branch_features(track, _starts(364), mel, N_FRAMES)
    return f[:300].contiguous(), f[300:].contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("n,batch", [(150, 64), (40, 16), (5, 64), (64, 64)])
def test_scoring_unchanged(model, prec, n, batch):
    """lsd_score_branch_features logits are bit for bit lsd_score_windows': several batches (pipelined on the bf16 route), a short
    last batch, one batch."""
    model.compute_precision = prec
    track, mel = _track(11)
    p = lb.Predictor(model, batch_size=batch)
    starts = _starts(n)
    a_from = [s + 2 for s in starts]
    plain = p.score_track_logits(track, starts, mel, N_FRAMES, audio_starts_from=a_from).cpu()
    lg, f = p.score_track_branch_features(track, starts, mel, N_FRAMES, audio_starts_from=a_from)
    assert f.shape == (n, 448) and f.dtype == torch.float32
    assert torch.equal(lg.cpu(), plain)
    assert torch.isfinite(f).all()


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_features_are_the_head_inputs(model, seed0_sd, prec):
    """The float64 head on the exported rows gives the returned logits; the slices are the oracle's cls / raw / delta / hf within the
    per-route tolerances of test_gpu_parity.py."""
    model.compute_precision = prec
    track, mel = _track(21)
    p = lb.Predictor(model, batch_size=4)
    starts = [0, 50, 123, 200, 368]
    lg, f = p.score_track_branch_features(track, starts, mel, N_FRAMES)
    lg, f = lg.cpu().numpy(), f.cpu().numpy()
    assert np.abs(ato.head(seed0_sd, f) - lg).max() <= 1e-5
    sel = [0, 4]
    video = torch.stack([track[starts[i]:starts[i] + 32].cpu() for i in sel]).permute(0, 4, 1, 2, 3).float() / 255.0
    m = mel.cpu()
    audio = torch.stack([m[:, :, P._audio_start(starts[i], TA_FULL, N_FRAMES):][:, :, :128] for i in sel])
    inter = {}
    orc.forward(seed0_sd, video, audio, inter=inter)
    tol = {"cls": 5e-5, "art_raw": 5e-5, "art_delta": 5e-5, "art_hf": 5e-5} if prec == "fp32" else \
          {"cls": 6e-3, "art_raw": 8e-3, "art_delta": 5e-3, "art_hf": 2.5e-3}
    for key, (lo, hi) in zip(("cls", "art_raw", "art_delta", "art_hf"), SL):
        assert _rel(f[sel, lo:hi], inter[key].numpy()) <= tol[key], key


@pytest.mark.gpu
@pytest.mark.parametrize("n,M", [(1, 1), (65, 7), (300, 64), (65, 256), (300, 1)])
def test_values_match_oracle(model, seed0_sd, feats300, n, M):
    f_all, extra = feats300
    feats = f_all[:n].contiguous()
    g = torch.Generator(device="cuda").manual_seed(M)
    src = torch.cat([extra, f_all[300 - M:]])[:M] if M <= 64 else f_all[torch.randperm(300, generator=g, device="cuda")[:M]]
    bg = src.contiguous()
    p = lb.Predictor(model)
    values, phi = p.branch_attribution(feats, bg)
    assert values.shape == (n, 16) and phi.shape == (n, 4)
    v, ph = values.cpu().numpy().astype(np.float64), phi.cpu().numpy().astype(np.float64)
    vref = ato.coalition_values(seed0_sd, feats.cpu().numpy(), bg.cpu().numpy())
    assert (np.abs(v - vref) <= 1e-5 * (1 + np.abs(vref))).all(), np.abs(v - vref).max()
    assert np.abs(ph - ato.shapley(vref)).max() <= 2e-5
    # v(15) is the plain logit of the window's head (the head kernel's logit of the same rows)
    plain = ato.head(seed0_sd, feats.cpu().numpy())
    assert np.abs(v[:, 15] - plain).max() <= 2e-5
    # efficiency to fp32 rounding
    eff = ph.sum(axis=1) - (v[:, 15] - v[:, 0])
    assert (np.abs(eff) <= 4e-6 * (1 + np.abs(v).max(axis=1))).all(), np.abs(eff).max()


@pytest.mark.gpu
def test_v15_is_the_scoring_logit(model):
    model.compute_precision = "bf16"
    track, mel = _track(31)
    p = lb.Predictor(model)
    lg, f = p.score_track_branch_features(track, _starts(70), mel, N_FRAMES)
    values, _ = p.branch_attribution(f, f[:9])
    assert float((values[:, 15] - lg).abs().max()) <= 2e-5


@pytest.mark.gpu
def test_exact_identities(model, feats300):
    f_all, _ = feats300
    p = lb.Predictor(model)
    for i in (0, 17, 299):
        x = f_all[i:i + 1]
        for bg in (x, torch.cat([x, x])):                          # one copy, and two (their sum halves exactly)
            values, phi = p.branch_attribution(x, bg.contiguous())
            assert (values == values[:, 15:16]).all() and (phi == 0).all()
        for q, (lo, hi) in enumerate(SL):                          # a background that differs in slice q only
            bg = x.clone()
            bg[:, lo:hi] = f_all[(i + 101) % 300, lo:hi]
            _, phi = p.branch_attribution(x, bg)
            others = [r for r in range(4) if r != q]
            assert (phi[0, others] == 0).all(), (i, q, phi)
            assert phi[0, q] != 0


@pytest.mark.gpu
def test_deterministic_and_split(model, feats300):
    f_all, extra = feats300
    p = lb.Predictor(model)
    bg = extra[:37].contiguous()
    v1, p1 = p.branch_attribution(f_all, bg)
    v2, p2 = p.branch_attribution(f_all, bg)
    assert torch.equal(v1, v2) and torch.equal(p1, p2)
    va, pa = p.branch_attribution(f_all[:111].contiguous(), bg)
    vb, pb = p.branch_attribution(f_all[111:].contiguous(), bg)
    assert torch.equal(torch.cat([va, vb]), v1) and torch.equal(torch.cat([pa, pb]), p1)


@pytest.mark.gpu
def test_c_abi_errors(model, feats300):
    f_all, extra = feats300
    L = _cabi.lib()
    n, M = 10, 4
    need = L.lsd_branch_attribution_workspace_bytes(n, M)
    assert need > 0
    for bad in [(-1, 4), (10, 0), (10, 257), (2 ** 20, 256)]:
        assert L.lsd_branch_attribution_workspace_bytes(*bad) == 0
    values = torch.full((n, 16), 7.0, device="cuda")
    phi = torch.full((n, 4), 7.0, device="cuda")
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    f, bg = f_all[:n].contiguous(), extra[:M].contiguous()
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        n0 = model.launch_count()

        def call(hp=h.ptr, fp=f.data_ptr(), nn=n, bp=bg.data_ptr(), mm=M, vp=values.data_ptr(), pp=phi.data_ptr(), wp=ws.data_ptr(),
                 wb=need):
            return L.lsd_branch_attribution(hp, fp, nn, bp, mm, vp, pp, wp, wb, None)

        assert call(hp=None) == _cabi.LSD_ERR_ARG
        assert call(fp=None) == _cabi.LSD_ERR_ARG
        assert call(bp=None) == _cabi.LSD_ERR_ARG
        assert call(vp=None) == _cabi.LSD_ERR_ARG
        assert call(pp=None) == _cabi.LSD_ERR_ARG
        assert call(wp=None) == _cabi.LSD_ERR_ARG
        assert call(nn=-1) == _cabi.LSD_ERR_SHAPE
        assert call(mm=0) == _cabi.LSD_ERR_SHAPE
        assert call(mm=257) == _cabi.LSD_ERR_SHAPE
        assert call(nn=2 ** 20, mm=256) == _cabi.LSD_ERR_SHAPE
        assert call(wb=need - 1) == _cabi.LSD_ERR_WORKSPACE
        assert model.launch_count() == n0
        assert (values == 7.0).all() and (phi == 7.0).all()
        bare = _cabi.Handle(0)                                          # no weights loaded
        assert call(hp=bare.ptr) == _cabi.LSD_ERR_WEIGHTS
        bare.close()
        n0 = model.launch_count()
        # feats_out NULL on the scoring entry
        track, mel = _track(3)
        lg = torch.empty(2, device="cuda")
        sw = L.lsd_score_workspace_bytes(h.ptr, 2, 32, 96, 96, 80, 128, model._precision())
        wsb = torch.empty(sw, dtype=torch.uint8, device="cuda")
        rc = L.lsd_score_branch_features(h.ptr, track.data_ptr(), N_FRAMES, 96, 96, (C.c_int32 * 2)(0, 5), None, 2, 32, mel.data_ptr(),
                                         80, TA_FULL, N_FRAMES, 128, model._precision(), 2, lg.data_ptr(), None, wsb.data_ptr(), sw, None)
        assert rc == _cabi.LSD_ERR_ARG
        assert model.launch_count() == n0
        assert call() == _cabi.LSD_OK
    torch.cuda.synchronize()
    assert torch.isfinite(values).all()


@pytest.mark.gpu
def test_attribution_track_and_long_video(model):
    """attribution_track on a track background and on a reference background, and the long-video entry equals attribution_track
    on the selected track."""
    model.compute_precision = "bf16"
    spec = SCENARIOS["one_track_localised_fake"]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(model)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, attribution=True)
    tr = next(t for t in tracks if int(t["track_id"]) == res["selected_track_id"])
    att = res["attribution"]
    crops, local = _track_u8(tr)
    crops = torch.from_numpy(np.ascontiguousarray(crops)).cuda()
    starts = [int(s) for s in tr["chunk_starts"]]
    want = pred.attribution_track(crops, local, torch.from_numpy(np.ascontiguousarray(mel, dtype=np.float32)).cuda(),
                                  n_frames, audio_starts_from=starts)
    assert json.dumps(att, sort_keys=True, default=str) == json.dumps(dict(want, track_id=res["selected_track_id"]), sort_keys=True,
                                                                      default=str)
    n = len(starts)
    assert att["background"] == "track" and att["background_size"] == min(n, 64) and att["window_starts"] == starts
    assert att["branches"] == list(ato.BRANCHES) and att["phi"].shape == (n, 4) and att["values"].shape == (n, 16)
    assert np.array_equal(att["base_logit"], att["values"][:, 0])
    assert att["frame_first"] == starts[0] and len(att["frame_timeline"]["sync"]) == starts[-1] + 32 - starts[0]
    ref = pred.attribution_track(crops, local, torch.from_numpy(np.ascontiguousarray(mel, dtype=np.float32)).cuda(),
                                 n_frames, background=torch.zeros(3, 448, device="cuda"), audio_starts_from=starts)
    assert ref["background"] == "reference" and ref["background_size"] == 3
    assert np.array_equal(ref["logits"], att["logits"])
