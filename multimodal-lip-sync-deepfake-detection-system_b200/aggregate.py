"""Window aggregation and decision gates of the long-video path: host mirror of the inline block of
`Predictor._predict_long_video` (app/inference/predictor.py:856-1155, verdict rule :1235).

Inputs are the per-window confidences this package's scorer returns plus the per-window speaking-activity and VAD
coverage values the reference computes on the host (`predictor.py:764-830`); output is the reference's decision
(`real` / `fake` / `uncertain`) with the same intermediate quantities and the same order of overrides.  O(#windows) numpy,
float32 where the reference uses float32.  Pinned against the real reference by tests/golden/verdict_golden.json.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Sequence

import numpy as np


def _robust(conf: Sequence[float], smoothing: str, trim_ratio: float) -> float:
    # predictor.py:246-260
    if not len(conf):
        return 0.5
    arr = np.asarray(conf, dtype=np.float32)
    if smoothing == "none":
        return float(arr.mean())
    if smoothing == "median":
        return float(np.median(arr))
    n = int(arr.size)
    k = int(n * trim_ratio)
    if k <= 0 or (2 * k) >= n:
        return float(arr.mean())
    return float(np.sort(arr)[k: n - k].mean())


def av_offset_profile(confs, valid, offsets: Sequence[int], smoothing: str = "median", trim_ratio: float = 0.1) -> Dict[str, Any]:
    """Sync profile of an audio-offset sweep.  `confs` / `valid`: (n_windows, K) calibrated confidences and the mask of entries
    whose audio slice needed no clamping; `offsets`: the K offsets (mel columns).  Per offset, the robust aggregate of the valid
    windows (`_robust`, the window aggregation of predictor.py:246-260) or None when no window is valid there.  `best_offset`:
    the argmax; ties go to the smaller |d|, then the smaller d.  `confidence_at_zero` / `margin` are None when offset 0 is
    not in the sweep or has no valid window."""
    conf = np.asarray(confs, dtype=np.float32).reshape(-1, len(offsets))
    ok = np.asarray(valid, dtype=bool).reshape(conf.shape)
    profile: List[Optional[float]] = []
    for k in range(len(offsets)):
        sel = conf[ok[:, k], k]
        profile.append(_robust(sel.tolist(), smoothing, trim_ratio) if sel.size else None)
    scored = [(p, int(d)) for p, d in zip(profile, offsets) if p is not None]
    best = max(scored, key=lambda pd: (pd[0], -abs(pd[1]), -pd[1])) if scored else None
    at_zero = next((p for p, d in zip(profile, offsets) if int(d) == 0), None)
    return {
        "offsets": [int(d) for d in offsets], "profile": profile, "n_valid": [int(x) for x in ok.sum(axis=0)],
        "best_offset": best[1] if best else None, "best_confidence": best[0] if best else None,
        "confidence_at_zero": at_zero,
        "margin": (best[0] - at_zero) if (best is not None and at_zero is not None) else None,
    }


def frame_evidence_timeline(starts: Sequence[int], temporal, segment_frames: int, T: int):
    """Per-frame timeline of occlusion evidence.  `starts`: first frame of every window; `temporal`: (n_windows, S) evidence of
    the window's frame segments [j*s, min((j+1)*s, T)), s = `segment_frames` (`Predictor.explain_track`).  Returns
    `(first_frame, values)`: values[f] belongs to frame first_frame + f, from the first window's start to the last window's end.
    A frame's value is the mean over every (window, segment) pair that covers it, None where no window covers it."""
    s, T = int(segment_frames), int(T)
    if not len(starts):
        return 0, []
    ev = np.asarray(temporal, dtype=np.float64).reshape(len(starts), -1)
    if ev.shape[1] != -(-T // s):
        raise ValueError(f"temporal has {ev.shape[1]} segments, {T} frames in segments of {s} make {-(-T // s)}")
    st = np.asarray(starts, dtype=np.int64)
    first = int(st.min())
    total = np.zeros(int(st.max()) + T - first, dtype=np.float64)
    count = np.zeros_like(total)
    seg_of = np.arange(T) // s                                       # segment of every frame of a window
    for i, a in enumerate(st - first):
        total[a:a + T] += ev[i, seg_of]
        count[a:a + T] += 1
    return first, [float(t / c) if c else None for t, c in zip(total, count)]


def columns_to_frames(first_col: int, values: Sequence[Optional[float]], Ta_full: int, total_v_frames: int):
    """A per-mel-column timeline (`values[c]` belongs to column first_col + c, None where nothing covers it) as a per-video-frame
    timeline.  Column c belongs to frame c * total_v_frames // Ta_full, in integers, the ratio `_audio_start` uses to place a
    window's audio.  Returns `(first_frame, frame_values)`, from the frame of the first column to the frame of the last one; a
    frame's value is the mean of its columns that are not None, None when it has none (also a frame no column maps to)."""
    Ta_full, nv = int(Ta_full), int(total_v_frames)
    if Ta_full < 1 or nv < 1:
        raise ValueError(f"Ta_full and total_v_frames must be >= 1, got {Ta_full} and {nv}")
    if not len(values):
        return 0, []
    cols = np.arange(int(first_col), int(first_col) + len(values), dtype=np.int64)
    frames = cols * nv // Ta_full
    first = int(frames[0])
    total = np.zeros(int(frames[-1]) - first + 1, dtype=np.float64)
    count = np.zeros_like(total)
    for f, v in zip(frames - first, values):
        if v is not None:
            total[f] += float(v)
            count[f] += 1
    return first, [float(t / c) if c else None for t, c in zip(total, count)]


BRANCHES = ("sync", "raw", "delta", "hf")


def branch_attribution_summary(phi, probs, confidence_threshold: float = 0.5, smoothing: str = "median", trim_ratio: float = 0.1,
                               starts: Optional[Sequence[int]] = None, T: int = 32) -> Dict[str, Any]:
    """Summary of branch attributions (`Predictor.attribution_track`).  `phi`: (n_windows, 4) Shapley values in logit space of the
    branches `BRANCHES` (> 0 pushes a window toward real); `probs`: (n_windows,) calibrated P(real).  A window is decided real when
    P(real) >= `confidence_threshold`.
      `mean_phi`, `median_phi` (4,): per branch over the windows;
      `share` (4,): each branch's mean |phi| over the sum of the four (zeros when every phi is 0);
      `leading_branch` (n,): per window, the branch with the most positive phi when it is decided real, the most negative when
        it is decided fake;
      `confidence`, `verdict`: the robust aggregate of `probs` (`_robust`, predictor.py:246-260) and its side of the threshold;
      `verdict_driver`: the branch whose mean phi pushes hardest toward that verdict (largest for "real", smallest for "fake");
        None without windows;
      `frame_first`, `frame_timeline`: with `starts` (first frame of every window, T frames each), per branch the per-frame mean
        of phi over the windows covering the frame (`frame_evidence_timeline` with one segment per window)."""
    p = np.asarray(phi, dtype=np.float64)
    if p.ndim != 2 or p.shape[1] != len(BRANCHES):
        raise ValueError(f"phi must be (n_windows, {len(BRANCHES)}), got shape {p.shape}")
    pr = np.asarray(probs, dtype=np.float64).reshape(-1)
    if pr.shape[0] != p.shape[0]:
        raise ValueError(f"probs has {pr.shape[0]} entries for {p.shape[0]} windows")
    thr = float(confidence_threshold)
    n = p.shape[0]
    mean_phi = p.mean(axis=0) if n else np.zeros(len(BRANCHES))
    median_phi = np.median(p, axis=0) if n else np.zeros(len(BRANCHES))
    mag = np.abs(p).mean(axis=0) if n else np.zeros(len(BRANCHES))
    share = mag / mag.sum() if mag.sum() > 0 else np.zeros(len(BRANCHES))
    real = pr >= thr
    leading = [BRANCHES[int(np.argmax(p[i]) if real[i] else np.argmin(p[i]))] for i in range(n)]
    conf = _robust(pr.tolist(), smoothing, trim_ratio)
    verdict = "real" if conf >= thr else "fake"
    driver = None
    if n:
        driver = BRANCHES[int(np.argmax(mean_phi) if verdict == "real" else np.argmin(mean_phi))]
    res = {"mean_phi": mean_phi, "median_phi": median_phi, "share": share, "leading_branch": leading, "confidence": conf,
           "verdict": verdict, "verdict_driver": driver}
    if starts is not None:
        if len(starts) != n:
            raise ValueError(f"starts has {len(starts)} entries for {n} windows")
        timeline = {}
        first = 0
        for b, name in enumerate(BRANCHES):
            first, timeline[name] = frame_evidence_timeline(starts, p[:, b:b + 1], int(T), int(T))
        res["frame_first"], res["frame_timeline"] = first, timeline
    return res


def augmentation_stability(probs, confidence_threshold: float = 0.5, smoothing: str = "median", trim_ratio: float = 0.1,
                           identity: int = 0) -> Dict[str, Any]:
    """Stability of a verdict under K variants of every window (`Predictor.robustness_track`).  `probs`: (n_windows, K) P(real);
    column `identity` is the unmodified window.  A window's decision is real when P(real) >= `confidence_threshold`.
      `confidence`: the robust aggregate (`_robust`, predictor.py:246-260) of the identity column;
      `variant_confidence` (K,): the same aggregate per variant;
      `tta_confidence`: the aggregate over windows of each window's mean P(real) over the variants;
      `window_spread` (n,): per window, the largest minus the smallest P(real) over the variants;
      `decision_flip_rate`: the fraction of (window, variant) entries whose decision differs from the identity's in that window;
      `verdict_stable`: every variant confidence lies on the same side of the threshold as `confidence`."""
    p = np.asarray(probs, dtype=np.float64)
    if p.ndim != 2 or not 0 <= int(identity) < p.shape[1]:
        raise ValueError(f"probs must be (n_windows, K) with column {identity} present, got shape {p.shape}")
    thr = float(confidence_threshold)
    conf = _robust(p[:, identity].tolist(), smoothing, trim_ratio)
    per_variant = [_robust(p[:, k].tolist(), smoothing, trim_ratio) for k in range(p.shape[1])]
    real = p >= thr
    return {
        "confidence": conf,
        "variant_confidence": per_variant,
        "tta_confidence": _robust(p.mean(axis=1).tolist(), smoothing, trim_ratio),
        "window_spread": p.max(axis=1) - p.min(axis=1),
        "decision_flip_rate": float((real != real[:, identity:identity + 1]).mean()) if p.size else 0.0,
        "verdict_stable": all((c >= thr) == (conf >= thr) for c in per_variant),
    }


def lowest_stable_quality(qualities: Sequence[Optional[int]], variant_confidence: Sequence[float], confidence: float,
                          threshold: float = 0.5) -> Optional[int]:
    """The lowest JPEG quality q such that every variant of quality >= q has its confidence on the same side of `threshold` as
    `confidence` (the plain window's; real when >= threshold).  Variants whose quality is None (uncompressed) are ignored.  None
    when the highest quality already lands on the other side, or when no variant has a quality.  A flip at some quality hides
    every lower quality, also those that land on the plain side again."""
    if len(qualities) != len(variant_confidence):
        raise ValueError(f"{len(qualities)} qualities for {len(variant_confidence)} variant confidences")
    side = float(confidence) >= float(threshold)
    by_q: Dict[int, bool] = {}
    for q, c in zip(qualities, variant_confidence):
        if q is not None:
            by_q[int(q)] = by_q.get(int(q), True) and ((float(c) >= float(threshold)) == side)
    lowest = None
    for q in sorted(by_q, reverse=True):
        if not by_q[q]:
            break
        lowest = q
    return lowest


def _speech_weighted(conf: Sequence[float], speaking: Sequence[float], vad: Optional[Sequence[float]], smoothing: str,
                     trim_ratio: float) -> float:
    # predictor.py:262-293
    if not len(conf):
        return 0.5
    if len(conf) != len(speaking):
        return _robust(conf, smoothing, trim_ratio)
    c = np.asarray(conf, dtype=np.float32)
    speech = np.clip(np.asarray(speaking, dtype=np.float32), 0.0, 1.0)
    if vad is not None and len(vad) == len(conf):
        combined = 0.7 * np.clip(np.asarray(vad, dtype=np.float32), 0.0, 1.0) + 0.3 * speech
    else:
        combined = speech
    weights = np.clip(0.2 + 0.8 * combined, 0.2, 1.0)
    denom = float(weights.sum())
    if denom <= 1e-8:
        return _robust(conf, smoothing, trim_ratio)
    return float(np.dot(c, weights) / denom)


def aggregate_long_video(
    window_confs: Sequence[float],
    window_speaking: Sequence[float],
    window_vad_weights: Optional[Sequence[float]] = None,
    mouth_check_result: str = "no_data",
    *,
    confidence_threshold: float = 0.5,
    confidence_smoothing: str = "median",
    trim_ratio: float = 0.1,
    weak_real_gate: float = 0.08,
    weak_real_window_threshold: float = 0.30,
    fake_vote_gate: float = 0.15,
    fake_vote_min_windows: int = 5,
    mouth_motion_check_enabled: bool = True,
    mouth_motion_fake_penalty: float = 0.10,
) -> Dict[str, Any]:
    """Decision for one video from its winning per-window results (ordered by time).

    `mouth_check_result` is the `check_result` of the reference's `_aggregate_mouth_motion_check`
    (`"likely_fake"`, `"uncertain"`, `"no_issue"`, `"no_data"`); defaults follow `Predictor.__init__` (predictor.py:60-76;
    note `Settings.fake_vote_gate` is 0.10, config.py:75 — pass it explicitly, SURVEY.md D10)."""
    thr = float(confidence_threshold)
    window_confs = [float(c) for c in window_confs]
    window_speaking = [float(s) for s in window_speaking]
    vad = [float(v) for v in window_vad_weights] if window_vad_weights is not None else None

    # ── median ⊕ speech-weighted blend (:871-879)
    window_median_confidence = _robust(window_confs, confidence_smoothing, trim_ratio)
    weighted_window_confidence = _speech_weighted(window_confs, window_speaking, vad, confidence_smoothing, trim_ratio)
    final_confidence = float(0.5 * window_median_confidence + 0.5 * weighted_window_confidence)

    conf_arr = np.asarray(window_confs, dtype=np.float32)
    speech_arr = np.asarray(window_speaking, dtype=np.float32)
    strong_real = int(np.sum(conf_arr >= max(thr + 0.15, 0.65)))
    strong_fake = int(np.sum(conf_arr <= min(thr - 0.15, 0.35)))
    mixed_window_signal = strong_real >= 2 and strong_fake >= 2

    # ── temporal confidence drift (:897-909)
    n_w = len(conf_arr)
    if n_w >= 4:
        half = n_w // 2
        first_half_avg = float(conf_arr[:half].mean())
        second_half_avg = float(conf_arr[half:].mean())
        temporal_drift = round(first_half_avg - second_half_avg, 4)
        temporal_confidence_drop = bool(temporal_drift >= 0.20)
    else:
        first_half_avg = second_half_avg = float(conf_arr.mean()) if n_w else float("nan")
        temporal_drift = 0.0
        temporal_confidence_drop = False

    # ── speech-weighted fake vote ratio (:929-947)
    if vad is not None and len(vad) == len(window_confs):
        vad_arr = np.clip(np.asarray(vad, dtype=np.float32), 0.0, 1.0)
        combined_speech_w = np.clip(0.7 * vad_arr + 0.3 * speech_arr, 0.0, 1.0)
    else:
        combined_speech_w = np.clip(speech_arr, 0.0, 1.0)
    speech_weights = np.clip(0.2 + 0.8 * combined_speech_w, 0.2, 1.0)
    fake_intensity = np.clip(thr - conf_arr, 0.0, 1.0)
    denom_w = float(speech_weights.sum())
    fake_vote_ratio = float(np.dot(speech_weights, fake_intensity) / denom_w) if denom_w > 1e-8 else 0.0
    fake_vote_ratio = float(np.clip(fake_vote_ratio / max(thr, 1e-6), 0.0, 1.0))

    # ── strict fake evidence: hard ratio + longest consecutive fake run (:963-983)
    speech_mask = speech_arr >= 0.45
    vote_src = conf_arr[speech_mask] if np.any(speech_mask) else conf_arr
    fake_ratio_hard = float(np.mean(vote_src < thr)) if vote_src.size else 0.0
    max_consec_fake = cur = 0
    for c in conf_arr:
        if c < thr:
            cur += 1
            max_consec_fake = max(max_consec_fake, cur)
        else:
            cur = 0
    strict_fake_evidence = bool(fake_ratio_hard >= 0.70 and max_consec_fake >= 8)

    # ── temporal-minority fake gate (:999-1019)
    meaningful_fake_evidence = fake_vote_ratio >= fake_vote_gate and strong_fake >= fake_vote_min_windows
    if meaningful_fake_evidence:
        fake_signal_confidence = float(1.0 - fake_vote_ratio)
        final_confidence = float(0.3 * final_confidence + 0.7 * fake_signal_confidence)
        final_confidence = min(final_confidence, thr - 1e-4)

    final_is_real = final_confidence >= thr
    window_consensus_uncertain = False
    override_reason: Optional[str] = None
    # ── mixed-consensus override (:1027-1032)
    if (not final_is_real) and mixed_window_signal and (not strict_fake_evidence):
        window_consensus_uncertain = True
        override_reason = "window_consensus_mixed"
        final_confidence = float(max(final_confidence, thr))
        final_is_real = True

    # ── sparse-real-signal guard (:1081-1105)
    max_window_conf = float(max(window_confs)) if window_confs else 0.0
    sparse_real_guard_applied = False
    if (not final_is_real) and max_window_conf >= weak_real_window_threshold and final_confidence < weak_real_gate:
        sparse_real_guard_applied = True
        override_reason = "sparse_real_signal"
        final_confidence = float(thr)
        final_is_real = True

    # ── mouth-motion result (:1116-1154)
    mouth_motion_override_applied = False
    if mouth_check_result != "no_data":
        if mouth_check_result == "likely_fake" and mouth_motion_check_enabled:
            final_confidence = float(max(0.0, final_confidence - mouth_motion_fake_penalty))
        elif mouth_check_result == "uncertain" and mouth_motion_check_enabled:
            if final_confidence < thr:
                mouth_motion_override_applied = True
                override_reason = override_reason or "mouth_motion_uncertain"
                final_confidence = float(thr)
        final_is_real = final_confidence >= thr

    verdict = "uncertain" if override_reason else ("real" if final_is_real else "fake")   # :1235
    return {
        "verdict": verdict,
        "is_real": bool(final_is_real),
        "is_fake": bool(not final_is_real),
        "confidence": float(final_confidence),
        "manipulation_probability": float(1.0 - final_confidence),
        "window_median_confidence": float(window_median_confidence),
        "window_weighted_confidence": float(weighted_window_confidence),
        "window_fake_vote_ratio": float(fake_vote_ratio),
        "strong_real_windows": strong_real,
        "strong_fake_windows": strong_fake,
        "window_consensus_uncertain": bool(window_consensus_uncertain),
        "strict_fake_evidence": bool(strict_fake_evidence),
        "sparse_real_guard_applied": bool(sparse_real_guard_applied),
        "mouth_motion_override_applied": bool(mouth_motion_override_applied),
        "override_reason": override_reason,
        "temporal_confidence_drop": bool(temporal_confidence_drop),
        "temporal_drift": round(temporal_drift, 4),
        "first_half_avg_confidence": round(first_half_avg, 4),
        "second_half_avg_confidence": round(second_half_avg, 4),
    }


def select_windows_by_time(tracks: List[Dict[str, Any]]) -> List[Dict[str, Any]]:
    """Per absolute start frame pick the track with the highest `0.75*window_conf + 0.25*stability`
    (predictor.py:765-789).  `tracks`: dicts with `track_id`, `stability`, `window_confidences`, `window_spans`."""
    by_start: Dict[int, List] = {}
    for tr in tracks:
        for i, span in enumerate(tr["window_spans"]):
            by_start.setdefault(int(span[0]), []).append((tr, i))
    out = []
    for abs_start in sorted(by_start):
        tr, i = max(by_start[abs_start], key=lambda t: 0.75 * float(t[0]["window_confidences"][t[1]]) + 0.25 * float(t[0].get("stability", 0.0)))
        out.append({"window_index": len(out), "frame_start": int(tr["window_spans"][i][0]), "frame_end": int(tr["window_spans"][i][1]),
                    "selected_track_id": int(tr["track_id"]), "confidence": float(tr["window_confidences"][i]), "chunk_index": i})
    return out
