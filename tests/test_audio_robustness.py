"""Audio robustness: `lsd_degrade_audio` (`Predictor.degrade_audio`) against the numpy restatement in oracle/audio_degrade_oracle.py,
`lsd_score_audio_clips` (`Predictor.score_track_audio_clips`) against `lsd_score_windows` on every clip alone, bit for bit,
`Predictor.audio_robustness_track` and the `audio_robustness` entry of `predict_long_video_from_tracks`."""
import ctypes as C
import json
import warnings

import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from lipsync_b200 import _cabi
from lipsync_b200.aggregate import lowest_stable_quality
from oracle import audio_degrade_oracle as orc
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


def _speech(n, seed=0, amp=0.3):
    """A speech-like test clip: a few harmonics under a syllable-rate envelope, plus a little hiss."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 16000.0
    f0 = 120 + 40 * np.sin(2 * np.pi * 0.7 * t)
    x = sum(np.sin(2 * np.pi * k * np.cumsum(f0) / 16000.0 + rng.uniform(0, 6)) / k for k in range(1, 8))
    env = 0.5 + 0.5 * np.sin(2 * np.pi * 4.0 * t) ** 2
    x = amp * env * x / np.max(np.abs(x)) + 0.003 * rng.standard_normal(n)
    return x.astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_oracle_mulaw_equals_audioop():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)
        import audioop
    s = np.arange(-32768, 32768, dtype=np.int16)
    assert np.array_equal(orc.lin2ulaw(s), np.frombuffer(audioop.lin2ulaw(s.tobytes(), 2), dtype=np.uint8))
    u = np.arange(256, dtype=np.uint8)
    assert np.array_equal(orc.ulaw2lin(u), np.frombuffer(audioop.ulaw2lin(u.tobytes(), 2), dtype=np.int16))


@pytest.mark.parametrize("n", [1, 2, 7, 40, 41, 100, 1001, 4096, 16001])
@pytest.mark.parametrize("rate", [8000, 4000])
def test_oracle_band_equals_resample_poly(n, rate):
    from scipy.signal import firwin, resample_poly
    x = np.random.default_rng(n).standard_normal(n)
    f = 16000 // rate
    ref = resample_poly(resample_poly(x, 1, f), f, 1)[:n]
    got = orc.band(x, rate)
    assert got.shape == (n,)
    assert np.max(np.abs(got - ref)) <= 1e-9 * np.max(np.abs(ref))
    assert np.max(np.abs(orc.kaiser_lowpass(f) - firwin(20 * f + 1, 1.0 / f, window=("kaiser", 5.0)))) <= 1e-15


@pytest.mark.parametrize("snr", [-20.0, 0.0, 10.0, 37.5, 60.0])
def test_oracle_noise_hits_the_snr(snr):
    x = _speech(24000, 1).astype(np.float64)
    y, g = orc.noise(x, snr, seed=7)
    assert np.allclose(y - x, g, rtol=0, atol=1e-15)
    assert abs(10 * np.log10(np.mean(x * x) / np.mean(g * g)) - snr) <= 0.01
    z, gz = orc.noise(np.zeros(100), snr, seed=7)                      # silence passes unchanged
    assert not z.any() and not gz.any()


@pytest.mark.parametrize("rt60", [0.05, 0.5, 1.3, 2.0])
def test_oracle_rir_length_decay_and_drr(rt60):
    h = orc.rir(rt60, seed=3)
    L = int(round(rt60 * 16000))
    assert len(h) == L and h[0] == 1.0
    assert abs(np.sum(h[1:] ** 2) - 1.0) <= 1e-12                        # direct-to-reverberant ratio 0 dB
    j = np.arange(1, L)
    env = h[1:] / orc.gaussian(3, orc.STREAM_RIR, j)                    # the decay without the noise: c 10^(-3 j / L)
    assert np.allclose(env / env[0], 10.0 ** (-3.0 * (j - 1) / L), rtol=1e-9)
    assert abs(20 * np.log10(env[-1] / env[0]) + 60.0 * (L - 2) / L) <= 1e-6   # 60 dB over the response


def test_oracle_generator_integers():
    """The two 24-bit integers of a draw are bit fields of one splitmix64 value; u1 is never 0 (the log is finite)."""
    r = orc.random_bits(5, 0, np.arange(10000))
    a, b = orc.uniforms24(5, 0, np.arange(10000))
    assert np.array_equal(a, (r >> np.uint64(40)).astype(np.int64)) and (a < 2 ** 24).all() and (b < 2 ** 24).all()
    assert np.isfinite(orc.gaussian(5, 0, np.arange(10000))).all()
    assert not np.array_equal(orc.random_bits(5, 1, np.arange(8)), orc.random_bits(5, 0, np.arange(8)))
    assert abs(np.mean(orc.gaussian(1, 0, np.arange(200000)) ** 2) - 1.0) < 0.02


def test_lowest_stable_snr_ladder():
    snr = [None, 30.0, 20.0, 10.0, 5.0, 0.0, None, None, None, None]
    conf = [0.8, 0.8, 0.7, 0.6, 0.4, 0.3, 0.2, 0.2, 0.9, 0.9]
    assert lowest_stable_quality(snr, conf, 0.8, 0.5) == 10               # 5 dB flips: the phone columns do not count
    assert lowest_stable_quality(snr, [0.8] * 10, 0.8, 0.5) == 0
    assert lowest_stable_quality(snr, [0.8, 0.3] + [0.8] * 8, 0.8, 0.5) is None
    assert lowest_stable_quality(snr, [0.2, 0.2, 0.2, 0.6, 0.2, 0.2] + [0.2] * 4, 0.2, 0.5) == 20   # fake side


def test_default_audio_degradation_variants():
    names, vs = lb.Predictor.audio_degradation_variants()
    assert names == ["none", "snr30", "snr20", "snr10", "snr5", "snr0", "phone", "noisy_phone", "reverb", "clipped"]
    assert vs[0] == {} and [v["snr_db"] for v in vs[1:6]] == [30, 20, 10, 5, 0]
    assert vs[6] == {"band_rate": 8000, "mulaw": True} and vs[7] == {"snr_db": 10, "band_rate": 8000, "mulaw": True}
    assert vs[8] == {"rt60": 0.5} and vs[9] == {"gain_db": 12}
    d = [lb.Predictor._degradation(k, v) for k, v in enumerate(vs)]
    A = _cabi
    assert [x.stages for x in d] == [0] + [A.LSD_AD_NOISE] * 5 + [A.LSD_AD_BAND | A.LSD_AD_MULAW,
                                                                 A.LSD_AD_NOISE | A.LSD_AD_BAND | A.LSD_AD_MULAW, A.LSD_AD_REVERB, A.LSD_AD_CLIP]
    t = lb.Predictor._degradation(0, (A.LSD_AD_REVERB | A.LSD_AD_CLIP, 0.3, 0.0, 6.0, 0, 9))
    assert (t.stages, round(t.rt60, 6), t.gain_db, t.seed) == (5, 0.3, 6.0, 9)


BAD_VARIANTS = [{"snr_db": float("nan")}, {"snr_db": -20.5}, {"snr_db": 61}, {"rt60": 0.04}, {"rt60": 2.5}, {"rt60": float("inf")},
                {"gain_db": -1}, {"gain_db": 41}, {"band_rate": 16000}, {"band_rate": 11025}, {"volume": 3}, {"seed": -1},
                (32, 0, 0, 0, 0, 0), (-1, 0, 0, 0, 0, 0), (1, 0.5, 0, 0, 0), (8, 0, 0, 0, 8001, 0)]


def test_argument_errors_without_gpu():
    p = lb.Predictor(None, device=torch.device("cpu"))
    x = np.zeros(1000, dtype=np.float32)
    for v in BAD_VARIANTS:
        with pytest.raises(ValueError):
            p.degrade_audio(x, [v])
    for vs in ([], [{}] * 65):
        with pytest.raises(ValueError):
            p.degrade_audio(x, vs)
    for bad in (np.zeros(0, dtype=np.float32), np.zeros((2, 100), dtype=np.float32)):
        with pytest.raises(ValueError):
            p.degrade_audio(bad, [{}])
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8)
    mels = torch.zeros((2, 80, 300))
    for args in ((track.float(), [0], mels), (track, [0], mels[0]), (track, [0], torch.zeros((0, 80, 300))),
                 (track, [0], torch.zeros((65, 80, 300))), (track, [40], mels)):
        with pytest.raises(ValueError):
            p.score_track_audio_clips(args[0], args[1], args[2], 64)
    with pytest.raises(ValueError):
        p.score_track_audio_clips(track, [0, 8], mels, 64, audio_starts_from=[0])
    with pytest.raises(ValueError):
        p.audio_robustness_track(track, [0], x, 64, variants=(["a", "b"], [{}]))


def test_long_video_audio_robustness_entry():
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    pred = lb.Predictor(None, device=torch.device("cpu"))
    fns = dict(score_fn=lambda tr: [0.7] * len(tr["chunk_starts"]), speech_fn=lambda tr, idxs: [0.6] * len(idxs),
               mouth_fn=lambda tr: {"check_result": "no_data"})
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, **fns)
    seen = []

    def audio_robustness_fn(tr):
        seen.append(int(tr["track_id"]))
        return {"confidence": 0.7, "lowest_stable_snr": 10}

    Ta_full = int(np.asarray(mel).shape[2])
    pcm = np.zeros(160 * (Ta_full - 1) + 37, dtype=np.float32)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, audio_robustness=True,
                                            audio_robustness_fn=audio_robustness_fn, pcm=pcm, **fns)
    assert "audio_robustness" not in base
    assert set(res) == set(base) | {"audio_robustness"}
    assert res["audio_robustness"]["track_id"] == res["selected_track_id"] == seen[0] and len(seen) == 1
    for k in base:                                                    # reported only: nothing else changes
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k
    for bad in (None, pcm[:-200], np.zeros(160 * Ta_full, dtype=np.float32)):
        with pytest.raises(ValueError):
            lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, audio_robustness=True,
                                              audio_robustness_fn=audio_robustness_fn, pcm=bad, **fns)
    assert len(seen) == 1


# ---------------------------------------------------------------------------------------------------------------- GPU
A = _cabi
STAGE_VARIANTS = [
    {},                                                   # 0 none
    {"mulaw": True},                                      # 1
    {"gain_db": 12.0},                                    # 2
    {"band_rate": 8000},                                  # 3
    {"band_rate": 4000},                                  # 4
    {"snr_db": 10.0, "seed": 3},                          # 5
    {"snr_db": -20.0, "seed": 1},                         # 6
    {"rt60": 0.5, "seed": 2},                             # 7
    {"rt60": 2.0, "seed": 5},                             # 8 the longest response, 32 000 taps
    {"band_rate": 8000, "mulaw": True},                   # 9 phone
    {"gain_db": 40.0, "mulaw": True},                     # 10
    {"snr_db": 37.5, "seed": 11},                         # 11
]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [16000 * 3 + 37, 16000 * 2, 40, 5])
def test_degrade_stages_against_oracle(model, n):
    p = lb.Predictor(model)
    x = _speech(n, 2)
    out = p.degrade_audio(torch.from_numpy(x).cuda(), STAGE_VARIANTS).cpu().numpy()
    assert out.shape == (len(STAGE_VARIANTS), n) and out.dtype == np.float32
    x64 = x.astype(np.float64)
    assert np.array_equal(out[0], x)
    assert np.array_equal(out[1], orc.mulaw(x))
    assert np.array_equal(out[2], orc.clip(x, 12.0))
    assert np.array_equal(out[10], orc.mulaw(orc.clip(x, 40.0)))
    for k, rate in ((3, 8000), (4, 4000)):
        assert np.max(np.abs(out[k] - orc.band(x64, rate))) <= 1e-5 * np.max(np.abs(x)), rate
    assert np.array_equal(out[9], orc.mulaw(out[3]))                   # phone: the mu-law of the device's own band output
    for k, snr, seed in ((5, 10.0, 3), (6, -20.0, 1), (11, 37.5, 11)):
        _, g = orc.noise(x64, snr, seed)
        d = out[k].astype(np.float64) - x64
        assert np.max(np.abs(d - g)) <= 1e-5, k
        assert abs(10 * np.log10(np.mean(x64 * x64) / np.mean(d * d)) - snr) <= 0.01, k
    for k, rt60, seed in ((7, 0.5, 2), (8, 2.0, 5)):
        ref = np.convolve(x64, orc.rir(rt60, seed))[:n]
        assert np.max(np.abs(out[k] - ref)) <= 1e-4 * np.sqrt(np.mean(ref * ref)), k


@pytest.mark.gpu
def test_degrade_chains_and_silence(model):
    """Four stages chained in one variant against the oracle's chain, and the fifth (mu-law) on top: bit for bit the mu-law of the
    device's own four-stage output.  A silent clip passes the noise stage unchanged.  The call is deterministic."""
    p = lb.Predictor(model)
    n = 16000 + 333
    x = _speech(n, 4, amp=0.6)
    v = {"rt60": 0.3, "snr_db": 15.0, "gain_db": 6.0, "band_rate": 4000, "seed": 21}
    out = p.degrade_audio(x, [v, dict(v, mulaw=True), v]).cpu().numpy()
    assert np.array_equal(out[0], out[2])
    ref = orc.degrade(x, 15, rt60=0.3, snr_db=15.0, gain_db=6.0, band_rate=4000, seed=21)
    assert np.max(np.abs(out[0] - ref)) <= 1e-4
    assert np.array_equal(out[1], orc.mulaw(out[0]))
    z = p.degrade_audio(np.zeros(5000, dtype=np.float32), [{"snr_db": 0.0}, {"snr_db": 60.0, "gain_db": 40.0}]).cpu().numpy()
    assert not z.any()


@pytest.mark.gpu
def test_degrade_argument_errors(model):
    """Bad arguments raise ValueError in Python; at the C-ABI they return LSD_ERR_SHAPE / LSD_ERR_ARG / LSD_ERR_WORKSPACE before
    anything is launched."""
    p = lb.Predictor(model)
    x = torch.zeros(1000, device="cuda")
    n0 = model.launch_count()
    for v in BAD_VARIANTS:
        with pytest.raises(ValueError):
            p.degrade_audio(x, [v])
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    out = torch.empty(2, 1000, device="cuda")
    need = L.lsd_degrade_audio_workspace_bytes(1000, 2)
    assert need > 0 and L.lsd_degrade_audio_workspace_bytes(0, 2) == 0 and L.lsd_degrade_audio_workspace_bytes(1000, 65) == 0
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")

    def call(vs, K=None, n=1000, pcm=x.data_ptr(), o=out.data_ptr(), ws_bytes=need):
        arr = (A.LsdAudioDegradation * max(1, len(vs)))(*[A.LsdAudioDegradation(*v) for v in vs]) if vs is not None else None
        return L.lsd_degrade_audio(h.ptr, pcm, n, arr, len(vs) if K is None else K, o, ws.data_ptr(), ws_bytes, None)

    ok = [(0, 0, 0, 0, 0, 0)]
    assert call(ok, K=0) == A.LSD_ERR_SHAPE
    assert call(ok * 65) == A.LSD_ERR_SHAPE
    assert call(ok, n=0) == A.LSD_ERR_SHAPE
    assert call(None, K=1) == A.LSD_ERR_ARG
    assert call(ok, pcm=None) == A.LSD_ERR_ARG
    assert call(ok, o=None) == A.LSD_ERR_ARG
    for bad in ((32, 0, 0, 0, 0, 0), (1, 0.01, 0, 0, 0, 0), (1, float("nan"), 0, 0, 0, 0), (2, 0, 61, 0, 0, 0),
                (2, 0, float("-inf"), 0, 0, 0), (4, 0, 0, -0.5, 0, 0), (4, 0, 0, 40.5, 0, 0), (8, 0, 0, 0, 16000, 0)):
        assert call([bad]) == A.LSD_ERR_ARG, bad
    assert call(ok * 2, ws_bytes=need - 1) == A.LSD_ERR_WORKSPACE
    assert call([(2, 0, float("nan"), 0, 0, 0)], K=1) == A.LSD_ERR_ARG
    assert model.launch_count() == n0
    assert call([(0, 0, float("nan"), 0, 0, 0)]) == A.LSD_OK          # parameters of stages a variant does not enable are ignored
    torch.cuda.synchronize()


def _track(seed, n_frames=200, H=96, W=96):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()


def _mels(seed, K, Ta_full, F=80):
    g = torch.Generator().manual_seed(seed)
    return (-80.0 * torch.rand((K, F, Ta_full), generator=g)).cuda()


def _per_clip(p, track, starts, mels, n_frames, **kw):
    return torch.stack([p.score_track_logits(track, starts, mels[k:k + 1], n_frames, **kw).cpu() for k in range(mels.shape[0])], dim=1)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_score_audio_clips_bitwise(model, prec):
    """Entry (i, k) is bit for bit lsd_score_windows on mels[k]: 9 windows in batches of 4, 4 and 1, computed and explicit audio
    starts."""
    model.compute_precision = prec
    track, mels = _track(71), _mels(72, 3, 800)
    n_frames = 200
    starts = list(range(0, n_frames - 32 + 1, 21))
    p = lb.Predictor(model, batch_size=4)
    out = p.score_track_audio_clips(track, starts, mels, n_frames).cpu()
    assert out.shape == (len(starts), 3) and out.dtype == torch.float32
    assert torch.equal(out, _per_clip(p, track, starts, mels, n_frames))
    frm = [s + 7 for s in starts]                                      # a span of a longer track: absolute frames for the audio
    out2 = p.score_track_audio_clips(track, starts, mels, n_frames + 7, audio_starts_from=frm).cpu()
    assert torch.equal(out2, _per_clip(p, track, starts, mels, n_frames + 7, audio_starts_from=frm))
    assert not torch.equal(out[:, 0], out[:, 1])


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 64])
def test_score_audio_clips_short_clip_and_k(model, K):
    """A clip of 100 columns under 128-column slices (every slice padded with its last column), at K = 1 and K = 64."""
    model.compute_precision = "bf16"
    track, mels = _track(73, n_frames=80), _mels(74, K, 100)
    starts = [0, 20, 48]
    p = lb.Predictor(model, batch_size=2)
    out = p.score_track_audio_clips(track, starts, mels, 80).cpu()
    assert torch.equal(out, _per_clip(p, track, starts, mels, 80))


@pytest.mark.gpu
def test_score_audio_clips_workspaces_and_fallback(model, monkeypatch):
    """Straight through the C-ABI in exactly the queried workspace and in twice it, batches of 3, 5 and 64: all equal.  On the
    launch-by-launch token path (LSD_TOK_FRONT=0) the rows go through lsd_score_windows and equal its per-clip logits on that path."""
    model.compute_precision = "bf16"
    track, mels = _track(75), _mels(76, 5, 700)
    n_frames, H, W = 200, 96, 96
    starts = list(range(0, 169, 21))
    K, n = 5, len(starts)
    L = _cabi.lib()
    p = lb.Predictor(model, batch_size=64)
    ref = _per_clip(p, track, starts, mels, n_frames)
    with model._lsd_lock:
        h = model._ensure_handle(model._device())
        for b in (3, 5, 64):
            need = L.lsd_score_audio_clips_workspace_bytes(h.ptr, b, K, 32, H, W, 80, 128, A.LSD_PREC_BF16)
            assert need > 0
            for ws_bytes in (need, 2 * need):
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
                L.lsd_workspace_invalidate(h.ptr)
                logits = torch.empty(n, K, dtype=torch.float32, device="cuda")
                rc = L.lsd_score_audio_clips(h.ptr, track.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*starts), None, n, 32, mels.data_ptr(),
                                             80, 700, n_frames, 128, K, A.LSD_PREC_BF16, b, logits.data_ptr(), ws.data_ptr(), ws_bytes,
                                             torch.cuda.current_stream().cuda_stream)
                _cabi.check(h.ptr, rc)
                assert torch.equal(logits.cpu(), ref), (b, ws_bytes)
                del ws
        L.lsd_workspace_invalidate(h.ptr)
    monkeypatch.setenv("LSD_TOK_FRONT", "0")
    p4 = lb.Predictor(model, batch_size=4)
    assert torch.equal(p4.score_track_audio_clips(track, starts, mels, n_frames).cpu(), _per_clip(p4, track, starts, mels, n_frames))


@pytest.mark.gpu
def test_score_audio_clips_argument_errors(model):
    model.compute_precision = "bf16"
    track = torch.zeros((64, 96, 96, 3), dtype=torch.uint8, device="cuda")
    mels = torch.zeros((2, 80, 300), device="cuda")
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    ws = model._workspace(1 << 20, track.device)
    out = torch.empty(2, 2, device="cuda")
    n0 = model.launch_count()

    def call(K=2, starts=(0, 8), mel_ptr=mels.data_ptr(), ws_bytes=ws.numel(), o=out.data_ptr()):
        return L.lsd_score_audio_clips(h.ptr, track.data_ptr(), 64, 96, 96, (C.c_int32 * 2)(*starts), None, 2, 32, mel_ptr, 80, 300, 64,
                                       128, K, A.LSD_PREC_BF16, 2, o, ws.data_ptr(), ws_bytes, None)

    assert call(K=0) == A.LSD_ERR_SHAPE
    assert call(K=65) == A.LSD_ERR_SHAPE
    assert call(starts=(0, 33)) == A.LSD_ERR_SHAPE
    assert call(starts=(-1, 0)) == A.LSD_ERR_SHAPE
    assert call(mel_ptr=None) == A.LSD_ERR_ARG
    assert call(o=None) == A.LSD_ERR_ARG
    assert call(ws_bytes=1024) == A.LSD_ERR_WORKSPACE
    assert model.launch_count() == n0


@pytest.mark.gpu
def test_audio_robustness_none_column(model):
    """lsd_logmel gives a clip the same bits alone and in a batch, so the `none` column of audio_robustness_track is bit for bit
    score_track_logits on the clean clip's log-mel; the report's fields follow from its logits."""
    from lipsync_b200.audio import logmel_db
    model.compute_precision = "bf16"
    n_frames = 200
    pcm = _speech(n_frames * 640, 9)                                     # 25 fps: 8 s
    x = torch.from_numpy(pcm).cuda()
    alone = logmel_db(x)
    batch = logmel_db(torch.stack([torch.zeros_like(x), x, 0.5 * x]))
    assert torch.equal(batch[1], alone)
    track = _track(77)
    starts = list(range(0, 169, 24))
    p = lb.Predictor(model, batch_size=16)
    res = p.audio_robustness_track(track, starts, pcm, n_frames)
    names, vs = p.audio_degradation_variants()
    assert res["variants"] == names and res["window_starts"] == starts
    assert res["snr_db"] == [None, 30.0, 20.0, 10.0, 5.0, 0.0, None, None, None, None]
    clean = p.score_track_logits(track, starts, alone[None], n_frames).cpu().tolist()
    assert res["confidence"] == p._robust_confidence([p._calibrate(float(v)) for v in clean])
    mels = logmel_db(p.degrade_audio(x, vs))
    logits = p.score_track_audio_clips(track, starts, mels, n_frames).cpu()
    assert logits[:, 0].tolist() == clean
    probs = np.array([[p._calibrate(float(v)) for v in row] for row in logits.tolist()])
    assert res["variant_confidence"] == [p._robust_confidence(probs[:, k].tolist()) for k in range(len(names))]
    assert res["lowest_stable_snr"] == lowest_stable_quality(res["snr_db"], res["variant_confidence"], res["confidence"], 0.5)


@pytest.mark.gpu
def test_long_video_audio_robustness_entry_on_gpu(model):
    model.compute_precision = "bf16"
    spec = SCENARIOS[sorted(SCENARIOS)[0]]
    tracks, n_frames = make_tracks(spec)
    mel, vad = make_audio(spec, n_frames)
    Ta_full = int(np.asarray(mel).shape[2])
    pcm = _speech(160 * (Ta_full - 1) + 80, 12)
    pred = lb.Predictor(model, batch_size=16)
    base = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames)
    res = lb.predict_long_video_from_tracks(pred, tracks, mel, vad, spec["fps"], n_frames, audio_robustness=True, pcm=pcm)
    assert set(res) == set(base) | {"audio_robustness"}
    ar = res["audio_robustness"]
    tr = next(t for t in tracks if int(t["track_id"]) == res["selected_track_id"])
    assert ar["track_id"] == res["selected_track_id"] and ar["window_starts"] == [int(s) for s in tr["chunk_starts"]]
    assert len(ar["variant_confidence"]) == 10
    for k in base:
        assert json.dumps(res[k], sort_keys=True, default=str) == json.dumps(base[k], sort_keys=True, default=str), k
