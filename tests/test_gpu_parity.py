"""Parity of the CUDA path (through the C-ABI) against the CPU oracle and the committed reference goldens.
Run on a B200: python -m pytest tests -m gpu.  Tolerances follow BASELINE.json: fp32 <= 1e-4 relative on logits,
bf16 <= 2e-2 absolute on logits, decisions (logit >= 0) identical."""
import numpy as np
import pytest
import torch

import lipsync_b200 as lb
from oracle import lipsync_oracle as orc
from oracle import logmel_oracle as lmo
from tests.golden.make_golden import CASES
from tests.golden.make_logmel_golden import CASES as MEL_CASES, make_pcm

pytestmark = pytest.mark.gpu

FP32_REL = 1e-4   # north_star: fp32 <= 1e-4 relative
BF16_ABS = 2e-2   # north_star: bf16 <= 2e-2 absolute on logits


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()


@pytest.fixture(scope="module")
def model(built, seed0_sd):
    m = lb.LipSyncModel()
    m.load_state_dict(seed0_sd, strict=True)
    return m.to("cuda:0").eval()


def _cl(x):  # oracle (B,C,T,H,W) / (B,C,H,W) -> channels-last flat
    if x.dim() == 5:
        return x.permute(0, 2, 3, 4, 1).contiguous().reshape(-1)
    if x.dim() == 4:
        return x.permute(0, 2, 3, 1).contiguous().reshape(-1)
    return x.contiguous().reshape(-1)


def _rel(a, b):
    return float((a - b).abs().max()) / max(1e-12, float(b.abs().max()))


@pytest.mark.parametrize("case", list(CASES))
def test_fp32_logits_match_reference_golden(model, golden, case):
    wseed, rescale, iseed, b, t, h, w, f, ta = CASES[case]
    sd = lb.make_synthetic_state_dict(wseed, rescale_head=rescale)
    model.load_state_dict(sd, strict=True)
    model.compute_precision = "fp32"
    video, audio = lb.synthetic_windows(iseed, b, t, h, w, f, ta)
    out = model(video.cuda(), audio.cuda()).cpu()
    ref = torch.from_numpy(golden[f"{case}/logits"])
    assert out.shape == (b,) and out.dtype == torch.float32
    assert _rel(out, ref) <= FP32_REL, (out, ref)
    assert ((out >= 0) == (ref >= 0)).all()
    model.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)


def test_fp32_stages_match_oracle(model, seed0_sd):
    model.compute_precision = "fp32"
    video, audio = lb.synthetic_windows(1, 2)
    inter = {}
    ref = orc.forward(seed0_sd, video, audio, inter=inter)
    out, aux = model(video.cuda(), audio.cuda(), return_aux=True)
    assert _rel(out.cpu(), ref) <= FP32_REL
    for name in ["v_stem", "v_layer1", "v_layer2", "v_layer3", "v_layer4", "a_stem", "a_layer1", "a_layer2", "a_layer3",
                 "a_layer4", "hf_front", "fused", "v_emb", "a_emb"]:
        got = model.stage(name).cpu()
        exp = _cl(inter[name])
        assert got.numel() == exp.numel(), name
        assert _rel(got, exp) <= 5e-5, (name, _rel(got, exp))
    tok = model.stage("t_layer3").cpu().view(2, 33, 256)
    assert _rel(tok, inter["t_layer3"]) <= 5e-5
    comb = model.stage("comb").cpu().view(2, 448)
    for i, key in enumerate(["art_raw", "art_delta", "art_hf"]):
        assert _rel(comb[:, 256 + 64 * i: 320 + 64 * i], inter[key]) <= 5e-5, key
    assert _rel(aux["cls_output"].cpu(), inter["cls"]) <= 5e-5
    assert _rel(aux["visual_tokens"].cpu(), inter["v_emb"]) <= 5e-5
    assert _rel(aux["audio_tokens"].cpu(), inter["a_emb"]) <= 5e-5
    assert _rel(aux["fused_tokens"].cpu(), inter["fused"]) <= 5e-5


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_batch_composition_independence_bitwise(model, prec):
    """Per-window results must not depend on the batch they ride in (sharding invariance, SURVEY.md §7.3)."""
    model.compute_precision = prec
    video, audio = lb.synthetic_windows(5, 3)
    v, a = video.cuda(), audio.cuda()
    full = model(v, a).cpu()
    one = model(v[1:2], a[1:2]).cpu()
    assert full[1].item() == one[0].item()
    rep = model(v.repeat(7, 1, 1, 1, 1), a.repeat(7, 1, 1, 1)).cpu()  # B = 21
    assert torch.equal(rep.view(7, 3), full.expand(7, 3))


def test_full_batch_64_property(model, golden):
    """BASELINE config 2 size (B=64): 16 copies of the 4 canonical windows reproduce the reference logits."""
    ref = torch.from_numpy(golden["canonical/logits"])
    video, audio = lb.synthetic_windows(1, 4)
    v = video.cuda().repeat(16, 1, 1, 1, 1)
    a = audio.cuda().repeat(16, 1, 1, 1)
    model.compute_precision = "fp32"
    out = model(v, a).cpu().view(16, 4)
    assert _rel(out, ref.expand(16, 4)) <= FP32_REL
    model.compute_precision = "bf16"
    out = model(v, a).cpu().view(16, 4)
    assert float((out - ref.expand(16, 4)).abs().max()) <= BF16_ABS
    assert ((out >= 0) == (ref.expand(16, 4) >= 0)).all()


@pytest.mark.parametrize("case", list(CASES))
def test_bf16_logits_within_budget(model, golden, case):
    wseed, rescale, iseed, b, t, h, w, f, ta = CASES[case]
    model.load_state_dict(lb.make_synthetic_state_dict(wseed, rescale_head=rescale), strict=True)
    model.compute_precision = "bf16"
    video, audio = lb.synthetic_windows(iseed, b, t, h, w, f, ta)
    out = model(video.cuda(), audio.cuda()).cpu()
    ref = torch.from_numpy(golden[f"{case}/logits"])
    model.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)
    assert float((out - ref).abs().max()) <= BF16_ABS, (out, ref)
    margin = ref.abs() > BF16_ABS  # decisions must agree wherever the reference is not inside the tolerance band
    assert ((out >= 0) == (ref >= 0))[margin].all()


def test_half_module_runs_tensor_core_path(model, golden):
    """predictor.py:196-197: model.half() + half inputs -> low-precision path, logits returned in the input dtype."""
    m = lb.LipSyncModel()
    m.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)
    m.half().to("cuda:0").eval()
    video, audio = lb.synthetic_windows(1, 4)
    out = m(video.cuda().half(), audio.cuda().half())
    assert out.dtype == torch.float16
    ref = torch.from_numpy(golden["canonical/logits"])
    assert float((out.float().cpu() - ref).abs().max()) <= BF16_ABS


def test_input_layouts_and_dtypes(model):
    model.compute_precision = "fp32"
    g = torch.Generator().manual_seed(11)
    u8 = torch.randint(0, 256, (2, 32, 96, 96, 3), generator=g, dtype=torch.uint8)
    _, audio = lb.synthetic_windows(9, 2)
    f_ncdhw = (u8.to(torch.float32) / 255.0).permute(0, 4, 1, 2, 3).contiguous()
    a = model(f_ncdhw.cuda(), audio.cuda()).cpu()
    b = model(u8.cuda(), audio.cuda(), video_layout="NDHWC").cpu()
    assert torch.equal(a, b)
    c = model(u8.permute(0, 4, 1, 2, 3).contiguous().cuda(), audio.cuda()).cpu()
    assert torch.equal(a, c)


def test_shape_errors_on_device(model):
    with pytest.raises(ValueError):
        model(torch.zeros(1, 3, 4, 96, 96, device="cuda"), torch.zeros(2, 1, 80, 128, device="cuda"))
    out = model(torch.zeros(0, 3, 32, 96, 96, device="cuda"), torch.zeros(0, 1, 80, 128, device="cuda"))
    assert out.shape == (0,)


def test_run_chunked_inference_matches_serial_oracle(model, seed0_sd):
    """The batched replacement of the serial loop (predictor.py:554-580) returns the same per-chunk confidences."""
    model.compute_precision = "fp32"
    g = torch.Generator().manual_seed(21)
    n_frames, stride = 32 + 8 * 5, 8
    track = torch.rand((3, n_frames, 96, 96), generator=g).numpy().astype(np.float32)
    starts = list(range(0, n_frames - 32 + 1, stride))
    chunks = [np.ascontiguousarray(track[:, s:s + 32]) for s in starts]
    mel_full = (-80.0 * torch.rand((1, 80, 500), generator=g)).numpy().astype(np.float32)
    p = lb.Predictor(model, batch_size=4)
    agg, confs = p._run_chunked_inference(chunks, starts, mel_full, n_frames)
    ref = []
    for c, s in zip(chunks, starts):
        a = p._align_audio_chunk(mel_full, s, n_frames)
        ref.append(float(torch.sigmoid(orc.forward(seed0_sd, torch.from_numpy(c)[None], torch.from_numpy(a)[None])).item()))
    assert len(confs) == len(starts) == 6
    assert np.abs(np.asarray(confs) - np.asarray(ref)).max() <= 2e-5
    assert abs(agg - float(np.median(np.asarray(ref, dtype=np.float32)))) <= 2e-5
    # variable-T forwards of _temporal_smoothed_confidence (T=16, Ta=64)
    r, cs, spans = p._temporal_smoothed_confidence(chunks[0], p._align_audio_chunk(mel_full, 0, n_frames))
    assert spans == [(0, 32), (0, 16), (8, 24), (16, 32)] and len(cs) == 4


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_score_track_device_window_builder(model, prec):
    """uint8 track -> device-built windows (lsd_score_windows) equals the host-built windows through forward()."""
    model.compute_precision = prec
    g = torch.Generator().manual_seed(31)
    n_frames = 32 + 8 * 9
    track = torch.randint(0, 256, (n_frames, 96, 96, 3), generator=g, dtype=torch.uint8)
    mel = -80.0 * torch.rand((1, 80, 650), generator=g)
    starts = list(range(0, n_frames - 32 + 1, 8))
    p = lb.Predictor(model, batch_size=4)  # 10 windows -> batches 4,4,2
    logits = p.score_track_logits(track.cuda(), starts, mel.cuda(), n_frames).cpu()
    vis = torch.stack([track[s:s + 32] for s in starts]).cuda()
    aud = torch.stack([torch.from_numpy(p._align_audio_chunk(mel.numpy(), s, n_frames)) for s in starts]).cuda()
    ref = model(vis, aud, video_layout="NDHWC").cpu()
    assert torch.equal(logits, ref)
    with pytest.raises(ValueError):
        p.score_track_logits(track.cuda(), [n_frames - 8], mel.cuda(), n_frames)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_long_video_decision_matches_oracle(model, seed0_sd, prec):
    """Decision level: per-window confidences from the CUDA scorer and from the CPU oracle lead to the same
    real / fake / uncertain verdict through the (reference-pinned) aggregation and gate block."""
    model.compute_precision = prec
    g = torch.Generator().manual_seed(41)
    n_win = 12
    n_frames = 32 + 8 * (n_win - 1)
    track = torch.randint(0, 256, (n_frames, 96, 96, 3), generator=g, dtype=torch.uint8)
    mel = -80.0 * torch.rand((1, 80, int(n_frames / 15 * 100)), generator=g)
    starts = list(range(0, n_frames - 32 + 1, 8))
    speaking = torch.rand(n_win, generator=g).tolist()
    vad = torch.rand(n_win, generator=g).tolist()
    p = lb.Predictor(model, batch_size=8)
    _, confs = p.score_track(track.cuda(), starts, mel.cuda(), n_frames)
    vis = torch.stack([track[s:s + 32] for s in starts]).permute(0, 4, 1, 2, 3).float() / 255.0
    aud = torch.stack([torch.from_numpy(p._align_audio_chunk(mel.numpy(), s, n_frames)) for s in starts])
    ref_confs = torch.sigmoid(orc.forward(seed0_sd, vis, aud)).tolist()
    tol = 1e-4 if prec == "fp32" else 5e-3   # on probabilities (sigmoid slope <= 1/4 of the logit tolerance)
    assert np.abs(np.asarray(confs) - np.asarray(ref_confs)).max() <= tol
    for gate in (0.15, 0.10):
        a = p.aggregate_long_video(confs, speaking, vad, "no_issue", fake_vote_gate=gate)
        b = p.aggregate_long_video(ref_confs, speaking, vad, "no_issue", fake_vote_gate=gate)
        assert a["verdict"] == b["verdict"] and a["override_reason"] == b["override_reason"]
        assert abs(a["confidence"] - b["confidence"]) <= 2 * tol


@pytest.mark.parametrize("name", list(MEL_CASES))
def test_logmel_matches_oracle(built, name):
    y = make_pcm(name)
    ref = lmo.preprocess_audio_pcm(y)
    out = lb.preprocess_audio_pcm(y)
    assert out.shape == ref.shape and out.dtype == np.float32
    assert out.max() == 0.0 and out.min() >= -80.0
    assert np.abs(out - ref).max() <= 2e-3  # dB; fp32 direct DFT vs pocketfft rFFT
    assert lb.preprocess_audio_pcm(y, target_frames=128).shape == (1, 80, 128)


def test_logmel_batched_clips_have_their_own_reference(built):
    ys = [make_pcm("noise_20480"), 0.01 * make_pcm("long_50000"), make_pcm("short_1000")]
    outs = lb.logmel_db([torch.from_numpy(y).cuda() for y in ys])
    for y, o in zip(ys, outs):
        ref = lmo.preprocess_audio_pcm(y)[0]
        assert np.abs(o.cpu().numpy() - ref).max() <= 2e-3


def test_logmel_equal_length_batch_matches_per_clip(built):
    """2-D `(B, n)` fast path == per-clip results, including clips whose PCM offset is not 16-byte aligned (n odd)."""
    g = torch.Generator().manual_seed(3)
    for n in (20480, 4001):
        pcm = (0.1 * torch.randn(5, n, generator=g)).cuda()
        pcm[2] *= 0.01
        batch = lb.logmel_db(pcm)
        assert batch.shape == (5, 80, 1 + n // 160)
        for i in range(5):
            ref = lmo.preprocess_audio_pcm(pcm[i].cpu().numpy())[0]
            assert np.abs(batch[i].cpu().numpy() - ref).max() <= 2e-3
            assert torch.equal(batch[i], lb.logmel_db(pcm[i].clone()))


def test_launch_counter_counts(model):
    model.compute_precision = "fp32"
    video, audio = lb.synthetic_windows(1, 1)
    n0 = model.launch_count()
    model(video.cuda(), audio.cuda())
    assert model.launch_count() - n0 > 50


def test_audio_encoder_subpath(model, seed0_sd):
    """lsd_audio_encoder == the audio branch of the full forward (bitwise) and == AudioEncoder.forward of the oracle
    (audio_encoder.py:173-205) within the bf16-route budget (split-bf16 operands: ~1e-4 relative)."""
    model.compute_precision = "bf16"
    video, audio = lb.synthetic_windows(1, 3)
    inter = {}
    orc.forward(seed0_sd, video, audio, inter=inter)
    _, aux = model(video.cuda(), audio.cuda(), return_aux=True)
    full = model.stage("a_feat").clone().view(3, -1, 256)
    got = model.encode_audio(audio.cuda())                    # (B, 256, T')
    assert got.shape == (3, 256, 16)
    assert torch.equal(got.transpose(1, 2).contiguous(), full)
    assert _rel(got.cpu(), orc.audio_encoder(seed0_sd, audio)) <= 2e-3
    # ragged / batch extremes of the sweep (BASELINE.json configs[2]): B = 1 and a non-multiple-of-tile batch
    for b in (1, 5):
        _, a = lb.synthetic_windows(7, b)
        o = model.encode_audio(a.cuda())
        assert o.shape == (b, 256, 16) and torch.isfinite(o).all()
    assert model.encode_audio(audio.cuda()[:0]).shape == (0, 256, 16)
    with pytest.raises(ValueError):
        model.encode_audio(audio.cuda()[:, 0])


def test_token_path_subpath(model, seed0_sd):
    """lsd_token_path (CrossModalAttention + TemporalTransformer, fusion_module.py:54-87 / temporal.py:79-111) fed with the
    projected embeddings of a full forward reproduces that forward's fused tokens and CLS output, and matches the oracle's
    `fused` / `cls` within the bf16-route budget."""
    model.compute_precision = "bf16"
    video, audio = lb.synthetic_windows(1, 3)
    inter = {}
    orc.forward(seed0_sd, video, audio, inter=inter)
    _, aux = model(video.cuda(), audio.cuda(), return_aux=True)
    fused, cls = model.fuse_tokens(aux["visual_tokens"], aux["audio_tokens"])
    # (same kernels; the full forward takes the cross-attention in-projections from the GEMM it merged with the feature
    #  projection — lsd_api.cu: pack_comb_proj —, the sub-path computes them from the embeddings: equal up to fp32 re-association
    #  in front of the fp16 operand rounding)
    assert _rel(fused, aux["fused_tokens"]) <= 1e-3
    assert _rel(cls, aux["cls_output"]) <= 1e-3
    f2, c2 = model.fuse_tokens(inter["v_emb"].cuda(), inter["a_emb"].cuda())
    assert _rel(f2.cpu(), inter["fused"]) <= 2e-3
    assert _rel(c2.cpu(), inter["cls"]) <= 2e-3
    # half windows (T=16, 8 audio tokens) and a large batch (BASELINE.json configs[3]: B=256)
    g = torch.Generator().manual_seed(4)
    v = torch.randn(256, 32, 256, generator=g).cuda()
    a = torch.randn(256, 16, 256, generator=g).cuda()
    fb, cb = model.fuse_tokens(v, a)
    f1, c1 = model.fuse_tokens(v[:5], a[:5])
    assert torch.equal(fb[:5], f1) and torch.equal(cb[:5], c1)      # batch-composition independence
    fh, ch = model.fuse_tokens(v[:4, :16], a[:4, :8])
    assert fh.shape == (4, 16, 256) and ch.shape == (4, 256) and torch.isfinite(ch).all()
    with pytest.raises(ValueError):
        model.fuse_tokens(v[:, :, :128], a)


@pytest.mark.parametrize("name", ["random_motion_random_audio", "static_face_loud_audio", "static_face_silent_audio",
                                  "speech_like_correlated", "slow_drift_anticorrelated", "short_audio_clamped_tail"])
def test_speech_stats_match_reference_golden(model, name):
    """Device speaking-alignment scores / mouth-motion statistics (lsd_track_motion + lsd_speech_stats) against the REAL
    reference functions (predictor.py:333-419) on the same synthetic tracks: score <= 2e-5 absolute, motion / energy at the
    reference's rounding (1e-6 / 1e-4), identical check results and aggregate."""
    import json, os
    from tests.golden.make_speech_golden import make_case
    with open(os.path.join(os.path.dirname(__file__), "golden", "speech_golden.json")) as fh:
        gold = json.load(fh)[name]
    track, starts, mel, n_frames = make_case(name)
    pred = lb.Predictor(model, batch_size=8)
    sp, mm, ae = pred.window_speech_stats(torch.from_numpy(track).cuda(), starts, torch.from_numpy(mel).cuda(), n_frames)
    assert np.abs(sp.cpu().numpy() - np.asarray(gold["speaking"], dtype=np.float64)).max() <= 2e-5
    checks = pred.mouth_motion_checks(mm.cpu().tolist(), ae.cpu().tolist())
    for got, exp in zip(checks, gold["mouth"]):
        assert abs(got["mouth_motion_energy"] - exp["mouth_motion_energy"]) <= 2e-6
        assert abs(got["audio_energy"] - exp["audio_energy"]) <= 2e-4
        assert got["check_result"] == exp["check_result"]
    agg = pred.aggregate_mouth_motion_checks(checks)
    assert agg["check_result"] == gold["aggregate"]["check_result"] and agg["samples_checked"] == gold["aggregate"]["samples_checked"]
    assert agg["counts"] == gold["aggregate"]["counts"]
    # single-window entry with the reference's own argument types: float32 (3,T,H,W) crop + (1,F,Ta) mel slice
    s0 = starts[1]
    visual = np.ascontiguousarray(track[s0:s0 + 32].transpose(3, 0, 1, 2)).astype(np.float32) / 255.0
    audio = pred._align_audio_chunk(mel, s0, n_frames)
    assert abs(pred._speaking_alignment_score(visual, audio) - gold["speaking"][1]) <= 2e-5


@pytest.mark.parametrize("name", ["speech_bursts", "continuous_noise", "near_silence", "short_clip", "loud_then_quiet"])
def test_vad_mask_matches_reference_golden(built, name):
    """Energy VAD (lsd_frame_energy + lsd_vad_mask + the reference's threshold rule) against the REAL
    `detect_voice_activity` (audio.py:105-245) on the same synthetic PCM: identical masks."""
    import json, os
    from tests.golden.make_vad_golden import make_pcm as vad_pcm
    with open(os.path.join(os.path.dirname(__file__), "golden", "vad_golden.json")) as fh:
        gold = json.load(fh)[name]
    mask, dur = lb.detect_voice_activity_pcm(vad_pcm(name))
    exp = np.asarray([c == "1" for c in gold["mask"]])
    assert mask.dtype == bool and mask.shape == exp.shape
    assert int((mask != exp).sum()) == 0
    assert abs(dur - gold["duration_sec"]) < 1e-9


def test_score_track_pipelined_batches_bitwise(model):
    """lsd_score_windows with a double workspace pipelines batches (tail of batch k on side streams while the main stream runs
    the encoder of batch k+1): logits must equal the single-batch result bit for bit, also when the two workspace halves are
    reused (5 batches) and when the last batch is ragged."""
    model.compute_precision = "bf16"
    g = torch.Generator().manual_seed(9)
    n_win = 19
    track = torch.randint(0, 256, (32 + 8 * (n_win - 1), 96, 96, 3), dtype=torch.uint8, generator=g).cuda()
    mel = (-80.0 * torch.rand(1, 80, 900, generator=g)).cuda()
    starts = [8 * i for i in range(n_win)]
    one = lb.Predictor(model, batch_size=32).score_track_logits(track, starts, mel, track.shape[0]).clone()
    for bs in (4, 8):
        piped = lb.Predictor(model, batch_size=bs).score_track_logits(track, starts, mel, track.shape[0]).clone()
        assert torch.equal(piped, one), bs
    again = lb.Predictor(model, batch_size=4).score_track_logits(track, starts, mel, track.shape[0])
    assert torch.equal(again, one)


@pytest.mark.parametrize("shape", [(2, 8, 72, 72, 80, 128), (1, 6, 50, 50, 40, 64), (3, 5, 100, 36, 80, 72)])
def test_bf16_odd_shapes_against_oracle(model, seed0_sd, shape):
    """Shapes that leave the fast paths: H not a multiple of the 16-row bands of the bulk-copy row kernel (72, 100), widths
    that are not multiples of 4 (50: direct-load fallback), odd stem widths (25: -inf edge of the max-pool), ragged T / Ta.
    bf16 budget on logits, same decisions unless the oracle logit is inside the budget of zero."""
    b, t, h, w, f, ta = shape
    model.compute_precision = "bf16"
    video, audio = lb.synthetic_windows(21, b, t, h, w, f, ta)
    ref = orc.forward(seed0_sd, video, audio)
    out = model(video.cuda(), audio.cuda()).float().cpu()
    assert float((out - ref).abs().max()) <= BF16_ABS, (out, ref)
    sure = ref.abs() > BF16_ABS
    assert ((out >= 0) == (ref >= 0))[sure].all()
    u8 = (video * 255).round().to(torch.uint8)
    out_u8 = model(u8.permute(0, 2, 3, 4, 1).contiguous().cuda(), audio.cuda(), video_layout="NDHWC").float().cpu()
    ref_u8 = orc.forward(seed0_sd, u8.float() / 255.0, audio)
    assert float((out_u8 - ref_u8).abs().max()) <= BF16_ABS


def test_scheduling_knobs_do_not_change_logits(model):
    """The side stream's SM share (LSD_SIDE_CTAS) only moves work between CTAs and streams: logits must be bit-identical to the
    default schedule.  The knob is read from the environment inside the library once per process, so each variant runs in a
    fresh interpreter."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import torch, hashlib, lipsync_b200 as lb\n"
            "m = lb.LipSyncModel(); m.load_state_dict(lb.make_synthetic_state_dict(0)); m.to('cuda:0').eval(); m.compute_precision = 'bf16'\n"
            "v, a = lb.synthetic_windows(33, 5)\n"
            "out = m(v.cuda(), a.cuda()).float().cpu()\n"
            "print('DIGEST', hashlib.sha256(out.numpy().tobytes()).hexdigest())\n") % root
    digests = {}
    for name, env in {"default": {}, "side_all_sms": {"LSD_SIDE_CTAS": "148"}}.items():
        # (LSD_STEM_RING=0: all variants run the flat shift-GEMM stem — the temporal-ring stem sums in a different order, it is
        #  compared with a tolerance in test_stem_ring_matches_flat_stem)
        r = subprocess.run([sys.executable, "-c", code], env={**os.environ, "LSD_STEM_RING": "0", **env}, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (name, r.stderr[-2000:])
        digests[name] = [l for l in r.stdout.splitlines() if l.startswith("DIGEST")][-1]
    assert len(set(digests.values())) == 1, digests


def test_stem_ring_matches_flat_stem(model):
    """The default stem (stem_ring.cu: three temporal taps as one N = 192 MMA over a TMEM ring of accumulators) against the flat
    shift-GEMM stem (LSD_STEM_RING=0): same bf16 operands, different fp32 summation order -> logits within a fraction of the bf16
    budget, for the canonical window, half windows (T=16) and a single frame (T=1: first step is also the last), in a fresh
    interpreter per route (the knob is read once per process)."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import torch, json, lipsync_b200 as lb\n"
            "m = lb.LipSyncModel(); m.load_state_dict(lb.make_synthetic_state_dict(0)); m.to('cuda:0').eval(); m.compute_precision = 'bf16'\n"
            "v, a = lb.synthetic_windows(41, 7)\n"
            "out = {}\n"
            "out['full'] = m(v.cuda(), a.cuda()).float().cpu().tolist()\n"
            "out['half'] = m(v[:, :, 8:24].contiguous().cuda(), a[..., 32:96].contiguous().cuda()).float().cpu().tolist()\n"
            "out['one'] = m(v[:3, :, :1].contiguous().cuda(), a[:3].cuda()).float().cpu().tolist()\n"
            "print('OUT', json.dumps(out))\n") % root
    res = {}
    for name, env in {"ring": {}, "flat": {"LSD_STEM_RING": "0"}}.items():
        r = subprocess.run([sys.executable, "-c", code], env={**os.environ, **env}, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (name, r.stderr[-2000:])
        res[name] = json.loads([l for l in r.stdout.splitlines() if l.startswith("OUT")][-1][4:])
    for k in res["ring"]:
        d = np.abs(np.asarray(res["ring"][k]) - np.asarray(res["flat"][k])).max()
        assert d <= 5e-3, (k, d, res["ring"][k], res["flat"][k])


def test_temporal_smoothed_confidence_values_match_oracle(model, seed0_sd):
    """predictor.py:295-331: the full window and the three half windows (T=16, T_a=64 -> 8 audio tokens lerped to 16) give the
    confidences the oracle computes for exactly those sub-windows, and their robust aggregate."""
    model.compute_precision = "fp32"
    g = torch.Generator().manual_seed(31)
    v = torch.rand((3, 32, 96, 96), generator=g).numpy().astype(np.float32)
    a = (-80.0 * torch.rand((1, 80, 128), generator=g)).numpy().astype(np.float32)
    p = lb.Predictor(model, batch_size=4)
    robust, confs, spans = p._temporal_smoothed_confidence(v, a)
    assert spans == [(0, 32), (0, 16), (8, 24), (16, 32)]
    ref = []
    for (v0, v1), (a0, a1) in zip(spans, [(0, 128), (0, 64), (32, 96), (64, 128)]):
        lg = orc.forward(seed0_sd, torch.from_numpy(np.ascontiguousarray(v[:, v0:v1]))[None], torch.from_numpy(np.ascontiguousarray(a[:, :, a0:a1]))[None])
        ref.append(float(torch.sigmoid(lg).item()))
    assert np.abs(np.asarray(confs) - np.asarray(ref)).max() <= 2e-5, (confs, ref)
    assert abs(robust - float(np.median(np.asarray(ref, dtype=np.float32)))) <= 2e-5
    model.compute_precision = "bf16"
    _, confs16, _ = p._temporal_smoothed_confidence(v, a)
    assert np.abs(np.asarray(confs16) - np.asarray(ref)).max() <= 5e-3    # 2e-2 on logits -> <= 5e-3 on probabilities


# Per-stage bounds of the tensor-core route (relative to the stage's largest magnitude), set at ~3x the measured deviation
# (profiles/r02_stage_errors.json): a compensating-error bug in one stage cannot hide behind the 2e-2 logit budget.
BF16_STAGE_BOUNDS = {"v_stem": 1.5e-2, "v_layer1": 2e-2, "v_layer2": 2e-2, "v_layer3": 2e-2, "v_layer4": 2e-2, "a_layer4": 1.5e-4,
                     "hf_front": 1.2e-2, "v_emb": 1e-2, "a_emb": 1.5e-4, "fused": 1.2e-2, "cls": 6e-3, "art_raw": 8e-3, "art_delta": 5e-3,
                     "art_hf": 2.5e-3}


def test_bf16_stages_match_oracle(model, seed0_sd):
    model.compute_precision = "bf16"
    video, audio = lb.synthetic_windows(1, 2)
    inter = {}
    ref = orc.forward(seed0_sd, video, audio, inter=inter)
    out, aux = model(video.cuda(), audio.cuda(), return_aux=True)
    assert float((out.cpu() - ref).abs().max()) <= BF16_ABS
    B = 2
    got = {
        "v_stem": model.planar_stage("x1", (B, 32, 24, 24, 64)),
        "v_layer1": model.planar_stage("y1", (B, 32, 24, 24, 64)),
        "v_layer2": model.planar_stage("y2", (B, 32, 12, 12, 128)),
        "v_layer3": model.planar_stage("y3", (B, 32, 6, 6, 256)),
        "v_layer4": model.planar_stage("y4", (B, 32, 3, 3, 256)),
        "a_layer4": model.planar_stage("ya4", (B, 1, 3, 16, 256), lo="ya4_lo"),
        "hf_front": model.planar_stage("hf_f", (B, 32, 48, 48, 32)),
        "v_emb": aux["visual_tokens"], "a_emb": aux["audio_tokens"], "fused": aux["fused_tokens"], "cls": aux["cls_output"],
    }
    comb = model.stage("comb").view(B, 448)
    for i, key in enumerate(["art_raw", "art_delta", "art_hf"]):
        got[key] = comb[:, 256 + 64 * i: 320 + 64 * i]
    errs = {}
    for name, g in got.items():
        exp = inter[name]
        exp = _cl(exp) if exp.dim() >= 4 else exp.reshape(-1)
        errs[name] = _rel(g.float().cpu().reshape(-1), exp)
    print("bf16 stage errors:", {k: f"{v:.2e}" for k, v in errs.items()})
    bad = {k: v for k, v in errs.items() if v > BF16_STAGE_BOUNDS[k]}
    assert not bad, (bad, errs)


def test_half_module_within_bf16_budget(model, golden):
    """f4: `.half()` module + half inputs (predictor.py:196-197, 217-219) stays inside the north-star low-precision budget."""
    m = lb.LipSyncModel()
    m.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)
    m.half().to("cuda:0").eval()
    video, audio = lb.synthetic_windows(1, 4)
    out = m(video.cuda().half(), audio.cuda().half())
    ref = torch.from_numpy(golden["canonical/logits"])
    assert float((out.float().cpu() - ref).abs().max()) <= BF16_ABS


def test_workspace_padding_survives_shape_changes(model):
    """ADVICE r1 (high): a pipelined lsd_score_windows call remembers the zero padding of BOTH workspace halves; a forward with
    other shapes through the same memory must invalidate them, or the next pipelined call convolves over stale padding."""
    model.compute_precision = "bf16"
    g = torch.Generator().manual_seed(41)
    n_frames = 32 + 8 * 11
    track = torch.randint(0, 256, (n_frames, 96, 96, 3), dtype=torch.uint8, generator=g).cuda()
    mel = (-80.0 * torch.rand((1, 80, 900), generator=g)).cuda()
    starts = [8 * i for i in range(12)]
    p = lb.Predictor(model, batch_size=4)          # 3 batches -> pipelined, both halves of the double workspace used
    first = p.score_track_logits(track, starts, mel, n_frames).clone()
    v, a = lb.synthetic_windows(9, 16)             # larger batch through the same workspace memory
    model(v.cuda(), a.cuda())
    again = p.score_track_logits(track, starts, mel, n_frames)
    assert torch.equal(first, again)
    vs, as_ = lb.synthetic_windows(9, 2, 16, 64, 64, 64, 100)   # other H/W/T as well
    model(vs.cuda(), as_.cuda())
    again = p.score_track_logits(track, starts, mel, n_frames)
    assert torch.equal(first, again)


def test_fused_token_kernels_match_layer_chain(model, seed0_sd):
    """tok_front.cu + tok_fused.cu (two launches, fp16 operands) against the launch-by-launch GEMM chain (split-bf16,
    LSD_TOK_FRONT=0 / LSD_TOK_FUSED=0) and the oracle — fused tokens (CrossModalAttention.forward, fusion_module.py:54-87) and
    CLS output (TemporalTransformer.forward, temporal.py:79-111) — and bitwise independence of a window from its slot /
    co-tenants in the CTA."""
    import os
    model.compute_precision = "bf16"
    g = torch.Generator().manual_seed(4)
    v = torch.randn(7, 32, 256, generator=g)
    a = torch.randn(7, 16, 256, generator=g)
    with torch.no_grad():
        f_ref = orc.cross_modal(seed0_sd, v, a)
        cls_ref = orc.temporal(seed0_sd, f_ref)
    res = {}
    try:
        for front, fused in (("0", "0"), ("1", "0"), ("0", "1"), ("1", "1")):
            os.environ["LSD_TOK_FRONT"], os.environ["LSD_TOK_FUSED"] = front, fused
            f, c = model.fuse_tokens(v.cuda(), a.cuda())
            res[front + fused] = (f.cpu(), c.cpu())
    finally:
        os.environ.pop("LSD_TOK_FRONT", None)
        os.environ.pop("LSD_TOK_FUSED", None)
    assert _rel(res["00"][0], f_ref) <= 5e-5 and _rel(res["00"][1], cls_ref) <= 2e-4          # chain
    assert _rel(res["10"][0], f_ref) <= 1e-3 and _rel(res["10"][1], cls_ref) <= 1e-3          # fused front alone
    assert torch.equal(res["01"][0], res["00"][0]) and _rel(res["01"][1], cls_ref) <= 2e-3    # fused transformer alone
    assert torch.equal(res["11"][0], res["10"][0]) and _rel(res["11"][1], cls_ref) <= 2e-3    # both (the default)
    f_all, c_all = model.fuse_tokens(v.cuda(), a.cuda())
    assert torch.equal(f_all.cpu(), res["11"][0]) and torch.equal(c_all.cpu(), res["11"][1])
    for i in range(7):
        fi, ci = model.fuse_tokens(v[i:i + 1].cuda(), a[i:i + 1].cuda())
        assert torch.equal(ci[0], c_all[i]) and torch.equal(fi[0], f_all[i])
    # half windows (16 + 1 tokens: four windows per CTA) and other lengths (slot 64 with 40 tokens, slot 32 with 29)
    for n, t, ta in ((5, 16, 8), (3, 40, 20), (3, 29, 16)):
        g2 = torch.Generator().manual_seed(100 + t)
        v2, a2 = torch.randn(n, t, 256, generator=g2), torch.randn(n, ta, 256, generator=g2)
        fh, ch = model.fuse_tokens(v2.cuda(), a2.cuda())
        with torch.no_grad():
            fh_ref = orc.cross_modal(seed0_sd, v2, a2)
            ch_ref = orc.temporal(seed0_sd, fh_ref)
        assert _rel(fh.cpu(), fh_ref) <= 1e-3 and _rel(ch.cpu(), ch_ref) <= 2e-3, (n, t, ta)


def test_cuda_graph_small_batch_path_bitwise(model):
    """`_infer_confidence` / `_temporal_smoothed_confidence` (predictor.py:212-244, 295-331) replay a captured CUDA graph for
    small host batches: same kernels, so the logits equal the launch-by-launch path bit for bit, also after the graph has been
    replayed with other data and after other shapes went through the handle."""
    model.compute_precision = "bf16"
    pg = lb.Predictor(model, use_cuda_graphs=True)
    pn = lb.Predictor(model, use_cuda_graphs=False)
    v, a = lb.synthetic_windows(3, 6)
    vs, as_ = [x.numpy() for x in v], [x.numpy() for x in a]
    for lo, n in ((0, 1), (1, 1), (0, 4), (2, 4), (5, 1)):
        assert pg._infer_logits(vs[lo:lo + n], as_[lo:lo + n]) == pn._infer_logits(vs[lo:lo + n], as_[lo:lo + n]), (lo, n)
    model(v.cuda(), a.cuda())                                   # other shapes through the shared handle in between
    r1, c1, s1 = pg._temporal_smoothed_confidence(vs[0], as_[0])
    r2, c2, s2 = pn._temporal_smoothed_confidence(vs[0], as_[0])
    assert c1 == c2 and r1 == r2 and s1 == s2
    assert len(pg._graphs) == 3                                  # (1 window), (4 windows), (3 half windows)


def test_score_batches_u8_transport_bitwise(model):
    """`Predictor.score_batches` on host fp32 windows (the `_run_chunked_inference` contract, predictor.py:554-580): windows whose
    pixels are exactly uint8 / 255.0 (video.py:552-556) cross PCIe as bytes and give the same logits, bit for bit, as the fp32
    upload and as a plain forward; windows that are not (here: one pixel nudged by an ulp) fall back to the fp32 upload."""
    model.compute_precision = "bf16"
    g = torch.Generator().manual_seed(5)
    _, a = lb.synthetic_windows(9, 10)
    v = torch.randint(0, 256, (10, 3, 32, 96, 96), dtype=torch.uint8, generator=g).to(torch.float32) / 255.0
    batches = [(v[0:4].contiguous(), a[0:4].contiguous()), (v[4:8].contiguous(), a[4:8].contiguous()),
               (v[6:10].contiguous(), a[6:10].contiguous()), (v[2:6].contiguous(), a[2:6].contiguous()), (v[8:10].contiguous(), a[8:10].contiguous())]
    ref = [model(vb.cuda(), ab.cuda()).float().cpu() for vb, ab in batches]
    p_u8 = lb.Predictor(model, host_transport="u8")
    p_f32 = lb.Predictor(model, host_transport="fp32")
    out_u8 = [t.clone() for t in p_u8.score_batches(batches)]
    assert p_u8.last_transport.startswith("u8") and p_u8.last_h2d_bytes_per_batch == 2 * 3 * 32 * 96 * 96 + 2 * 80 * 128 * 4
    out_f32 = [t.clone() for t in p_f32.score_batches(batches)]
    assert p_f32.last_transport == "fp32"
    for r, x, y in zip(ref, out_u8, out_f32):
        assert torch.equal(r, x) and torch.equal(r, y)
    # split transport (half of every batch as fp32 over PCIe, the rest packed and expanded on the device by lsd_expand_u8): same bits
    p_split = lb.Predictor(model, host_transport="u8", host_split=0.5)
    out_split = [t.clone() for t in p_split.score_batches(batches)]
    assert "split" in p_split.last_transport and p_split.last_h2d_bytes_per_batch == (4 + 1) * 3 * 32 * 96 * 96 + 2 * 80 * 128 * 4
    for r, x in zip(ref, out_split):
        assert torch.equal(r, x)
    # not k/255 data: detected, shipped as fp32, still identical to the plain forward
    v2 = v.clone()
    v2[5, 1, 7, 3, 2] = torch.nextafter(v2[5, 1, 7, 3, 2], torch.tensor(2.0))
    b2 = [(v2[0:4].contiguous(), a[0:4].contiguous()), (v2[4:8].contiguous(), a[4:8].contiguous()), (v2[6:10].contiguous(), a[6:10].contiguous())]
    ref2 = [model(vb.cuda(), ab.cuda()).float().cpu() for vb, ab in b2]
    out2 = [t.clone() for t in p_u8.score_batches(b2)]
    assert p_u8.last_transport == "fp32"
    for r, x in zip(ref2, out2):
        assert torch.equal(r, x)


def test_expand_u8_is_the_reference_division_bitwise():
    """`lsd_expand_u8`: device bytes -> fl(k / 255.0f), bit for bit the reference's `astype(np.float32) / 255.0` (video.py:552-556)
    for every k, at any 16-byte-aligned length; misaligned or odd-length arguments are refused."""
    from lipsync_b200 import _cabi
    L = _cabi.lib()
    g = torch.Generator().manual_seed(3)
    for n in (16, 256, 4096 + 16, 3 * 96 * 96):
        k = torch.randint(0, 256, (n,), dtype=torch.uint8, generator=g)
        k[:min(n, 256)] = torch.arange(min(n, 256), dtype=torch.uint8)
        src = k.cuda()
        dst = torch.full((n + 4,), -1.0, dtype=torch.float32, device="cuda")
        assert L.lsd_expand_u8(src.data_ptr(), dst.data_ptr(), n, torch.cuda.current_stream().cuda_stream) == _cabi.LSD_OK
        exp = torch.from_numpy(k.numpy().astype(np.float32) / 255.0)
        assert torch.equal(dst[:n].cpu(), exp) and bool((dst[n:] == -1.0).all())
    assert L.lsd_expand_u8(src.data_ptr(), dst.data_ptr(), 0, None) == _cabi.LSD_OK
    assert L.lsd_expand_u8(src.data_ptr(), dst.data_ptr(), 24, None) == _cabi.LSD_ERR_ARG
    assert L.lsd_expand_u8(src.data_ptr() + 1, dst.data_ptr(), 16, None) == _cabi.LSD_ERR_ARG
    assert L.lsd_expand_u8(None, dst.data_ptr(), 16, None) == _cabi.LSD_ERR_ARG


def test_preprocessed_validation_driver(model, seed0_sd, tmp_path):
    """The reference's preprocessed-mode evaluator (scripts/validate_pipeline.py:382-525) on this backend: confidences equal
    sigmoid(model(batch)) of the same batches bit for bit, decisions equal the fp32 oracle's, files are written."""
    model.compute_precision = "bf16"
    v, a = lb.synthetic_windows(21, 7)
    labels = torch.tensor([1, 0, 1, 1, 0, 0, 1])

    class DS:
        def __len__(self):
            return 7

        def get_item(self, idx, train_mode_override=False):
            return (None if idx == 2 else (v[idx], a[idx], labels[idx].float()))

    res = lb.run_preprocessed_validation(DS(), lb.Predictor(model), output_dir=str(tmp_path), batch_size=4)
    keep = [0, 1, 3, 4, 5, 6]
    assert [r["sample_idx"] for r in res["rows"]] == keep
    direct = torch.cat([model(v[[0, 1, 3]].cuda(), a[[0, 1, 3]].cuda()), model(v[[4, 5, 6]].cuda(), a[[4, 5, 6]].cuda())]).float().cpu()
    conf = torch.tensor([r["confidence"] for r in res["rows"]], dtype=torch.float64)
    assert torch.equal(conf, torch.sigmoid(direct).double())
    ref = orc.forward(seed0_sd, v[keep], a[keep])
    assert [r["predicted_label"] for r in res["rows"]] == [0 if float(torch.sigmoid(x)) >= 0.5 else 1 for x in ref]
    assert res["metrics"]["total_samples"] == 6 and (tmp_path / "predictions.csv").is_file() and (tmp_path / "metrics.json").is_file()
