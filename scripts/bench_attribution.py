"""Branch attribution on one GPU.  Two measurements in one run:
  * `Predictor.branch_attribution` on the exported head inputs of 1600 windows of one track, against M = 64 and M = 256
    background rows: ms per call and coalition rows per second, n * (15 M + 1) rows per call, and per kernel (torch.profiler);
  * `lsd_score_branch_features` against `lsd_score_windows` (`score_track_branch_features` / `score_track_logits`) on the same
    1600 windows, bf16 tensor-core route, batch 64 with the double (pipelined) workspace, inputs resident on the device.
Prints one JSON line (also written to --out).

Timing: CUDA events around blocks of back-to-back calls of >= --window-s seconds after warm-up; the calls alternate block by block
so all see the same clocks; the median block is reported.  The track (12 824 frames, 355 MB) is larger than the 126 MB L2; the
attribution inputs (2.9 MB of features) and the head's weights stay in L2.  The FLOP count of a call is the tail's
2 * (256 * 128 + 128 * 128) per coalition row plus the projections' 2 * (448 * 256 + 256 * 128) per window and background row.
The card's name, power limit and max SM clock are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lipsync_b200 as lb  # noqa: E402


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
    ap.add_argument("--windows", type=int, default=1600)
    ap.add_argument("--backgrounds", default="64,256")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--window-s", type=float, default=1.5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(gpu_info())
    model = lb.LipSyncModel()
    model.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)
    model.to("cuda:0").eval()
    model.compute_precision = "bf16"
    p = lb.Predictor(model, batch_size=64)
    T, H, W, stride = 32, 96, 96, 8
    n = a.windows
    n_frames = (n - 1) * stride + T
    g = torch.Generator().manual_seed(0)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    mel = (-80.0 * torch.rand((1, 80, int(n_frames * 100 / 25)), generator=g)).cuda()
    starts = [i * stride for i in range(n)]
    Ms = [int(x) for x in a.backgrounds.split(",")]
    with torch.no_grad():
        logits, feats = p.score_track_branch_features(track, starts, mel, n_frames)
        bitwise = bool(torch.equal(logits, p.score_track_logits(track, starts, mel, n_frames)))
        bgs = {M: feats[torch.tensor(p.track_background_index(n, M), device="cuda")].contiguous() for M in Ms}
        plain = lambda: p.score_track_logits(track, starts, mel, n_frames)  # noqa: E731
        with_feats = lambda: p.score_track_branch_features(track, starts, mel, n_frames)  # noqa: E731
        attr = {M: (lambda M=M: p.branch_attribution(feats, bgs[M])) for M in Ms}
        for _ in range(2):
            plain()
            with_feats()
            for M in Ms:
                attr[M]()
        torch.cuda.synchronize()
        tp, tf, ta = [], [], {M: [] for M in Ms}
        for _ in range(a.reps):
            tp.append(time_block(plain, a.window_s))
            tf.append(time_block(with_feats, a.window_s))
            for M in Ms:
                ta[M].append(time_block(attr[M], a.window_s / 2))
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        kern = {}
        for M in Ms:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    attr[M]()
                torch.cuda.synchronize()
            for name in ("branch_project_kernel", "coalition_tail_kernel", "attribution_finalize_kernel"):
                us = [ev.device_time_total or ev.time_range.elapsed_us() for ev in prof.events() if name in ev.name]
                kern[f"M{M}_{name}_us"] = round(median(us), 1) if us else None
    res.update({"windows": n, "batch": p.batch_size, "logits_bitwise_equal": bitwise,
                "plain_ms": round(median(tp), 3), "branch_features_ms": round(median(tf), 3),
                "branch_features_over_plain": round(median(tf) / median(tp), 4),
                "plain_ms_all": [round(x, 3) for x in tp], "branch_features_ms_all": [round(x, 3) for x in tf]})
    for M in Ms:
        rows = n * (15 * M + 1)
        flop = rows * 2 * (256 * 128 + 128 * 128) + (n + M) * 2 * (448 * 256 + 256 * 128)
        ms = median(ta[M])
        res.update({f"M{M}_rows": rows, f"M{M}_ms": round(ms, 3), f"M{M}_ms_all": [round(x, 3) for x in ta[M]],
                    f"M{M}_rows_per_s": round(rows / (ms * 1e-3), 1), f"M{M}_tflops": round(flop / (ms * 1e-3) / 1e12, 2)})
    res.update(kern)
    res["timing"] = (f"CUDA events, blocks of >= {a.window_s} s (attribution: {a.window_s / 2} s) after warm-up, alternating, median of "
                     f"{a.reps}; kernels: torch.profiler over 3 calls per M, median launch")
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    assert bitwise, "lsd_score_branch_features logits differ from lsd_score_windows"


if __name__ == "__main__":
    main()
