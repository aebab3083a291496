"""Audio robustness on one GPU.
1. Scoring: `Predictor.score_track_audio_clips` with K = 10 clip log-mels (64 windows x 10 = 640 rows, the shared-visual route)
   against `Predictor.score_track_logits` on the same 640 (window, clip) rows through the plain path (640 windows of the same
   uint8 track), bf16 tensor-core route, inputs resident on the device, batch 64.
2. Front end: `Predictor.degrade_audio` with the K = 10 `audio_degradation_variants` on a 60 s clip, then `audio.logmel_db` of the
   10 copies, and `degrade_audio` per stage on its own (one variant per call: none, noise, clip, band 8 kHz, band + mu-law, reverb
   at rt60 0.5 s and 2.0 s).  The reverb FIR's multiply-adds are counted from its length (n x L, less the triangle at the start);
   its rate is that count over the measured time of its call, which also includes one copy of the impulse response.
Timing: CUDA events around blocks of back-to-back calls of >= --window-s seconds after warm-up, the calls of a comparison
alternating block by block; the median block is reported.  The card's name, power limit and max SM clock are read in the same run.
Prints one JSON line (also written to --out)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lipsync_b200 as lb  # noqa: E402
from lipsync_b200.audio import logmel_db  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "clocks_max_sm": clock}


def time_block(fn, window_s):
    """ms per call of fn over a block of back-to-back calls lasting at least window_s (count sized from a probe)."""
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    e.record()
    e.synchronize()
    n = max(3, int(window_s * 1e3 / max(s.elapsed_time(e), 1e-3)))
    s.record()
    for _ in range(n):
        fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / n


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=64)
    ap.add_argument("--clip-s", type=float, default=60.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(gpu_info())
    model = lb.LipSyncModel()
    model.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)
    model.to("cuda:0").eval()
    model.compute_precision = "bf16"
    p = lb.Predictor(model, batch_size=64)
    names, variants = p.audio_degradation_variants()
    K = len(names)
    T, H, W, stride = 32, 96, 96, 8
    rows = a.windows * K
    n_frames = (rows - 1) * stride + T
    g = torch.Generator().manual_seed(0)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    ta_full = int(n_frames * 100 / 25)
    mel = (-80.0 * torch.rand((1, 80, ta_full), generator=g)).cuda()
    mels = (-80.0 * torch.rand((K, 80, ta_full), generator=g)).cuda()
    plain_starts = [i * stride for i in range(rows)]
    starts = plain_starts[:: max(1, rows // a.windows)][: a.windows]
    plain = lambda: p.score_track_logits(track, plain_starts, mel, n_frames)  # noqa: E731
    clips = lambda: p.score_track_audio_clips(track, starts, mels, n_frames)  # noqa: E731

    n = int(a.clip_s * 16000)
    t = np.arange(n) / 16000.0
    pcm = torch.from_numpy((0.3 * np.sin(2 * np.pi * 180 * t) * (0.5 + 0.5 * np.sin(2 * np.pi * 4 * t) ** 2)).astype(np.float32)).cuda()
    front = lambda: logmel_db(p.degrade_audio(pcm, variants))  # noqa: E731
    stage_variants = {"none": {}, "noise": {"snr_db": 10.0}, "clip": {"gain_db": 12.0}, "band8k": {"band_rate": 8000},
                      "phone": {"band_rate": 8000, "mulaw": True}, "reverb_0.5s": {"rt60": 0.5}, "reverb_2.0s": {"rt60": 2.0}}
    stage_fns = {k: (lambda v=v: p.degrade_audio(pcm, [v])) for k, v in stage_variants.items()}
    with torch.no_grad():
        for _ in range(2):
            plain()
            clips()
            front()
            for f in stage_fns.values():
                f()
        torch.cuda.synchronize()
        out = clips().cpu()
        ref = torch.stack([p.score_track_logits(track, starts, mels[k:k + 1], n_frames).cpu() for k in range(K)], dim=1)
        bitwise = bool(torch.equal(out, ref))
        tp, tc, tf = [], [], []
        ts = {k: [] for k in stage_fns}
        for _ in range(a.reps):
            tp.append(time_block(plain, a.window_s))
            tc.append(time_block(clips, a.window_s))
            tf.append(time_block(front, a.window_s))
            for k, f in stage_fns.items():
                ts[k].append(time_block(f, a.window_s / 4))
    res.update({
        "windows": a.windows, "variants": K, "variant_names": names, "rows_per_call": rows, "batch": p.batch_size,
        "plain_rows_per_s": round(rows / (median(tp) * 1e-3), 1), "clips_rows_per_s": round(rows / (median(tc) * 1e-3), 1),
        "plain_ms_all": [round(x, 3) for x in tp], "clips_ms_all": [round(x, 3) for x in tc],
        "clips_over_plain": round(median(tp) / median(tc), 3),
        "clips_bitwise_equal_per_clip_plain": bitwise,
        "clip_s": a.clip_s, "samples": n,
        "degrade_logmel_k10_ms": round(median(tf), 3), "degrade_logmel_k10_ms_all": [round(x, 3) for x in tf],
        "stage_ms": {k: round(median(v), 3) for k, v in ts.items()},
    })
    for k, rt60 in (("reverb_0.5s", 0.5), ("reverb_2.0s", 2.0)):
        L = int(round(rt60 * 16000))
        macs = n * L - L * (L - 1) / 2
        res[f"{k}_gmac"] = round(macs / 1e9, 3)
        res[f"{k}_gmac_per_s"] = round(macs / (median(ts[k]) * 1e-3) / 1e9, 1)
    res["timing"] = (f"CUDA events, blocks of >= {a.window_s} s (stages: {a.window_s / 4} s) after warm-up, alternating, median of "
                     f"{a.reps}; inputs resident on the device")
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    assert bitwise, "lsd_score_audio_clips differs from lsd_score_windows per clip"


if __name__ == "__main__":
    main()
