"""Crop-jitter robustness on one GPU: `Predictor.score_track_warps` with the K=12 variants of `robustness_track` (64 windows x 12
= 768 rows) against `Predictor.score_track_logits` on 768 plain windows of the same uint8 track, bf16 tensor-core route, inputs
resident on the device, batch 64 with the double (pipelined) workspace.  Prints one JSON line (also written to --out).

Timing: CUDA events around blocks of back-to-back calls of >= --window-s seconds after warm-up; the two calls alternate block
by block so both see the same clocks; the median block is reported as rows per second.  The track (6 168 frames, 171 MB)
exceeds the 126 MB L2.  A separate torch.profiler pass then times the builder kernel itself (`warp_windows_kernel`) and sets it
against the bytes it must move: 2 x rows x T x H x W x 3 (every source frame read once, every warped frame written once) over
the HBM bandwidth of the data sheet (7.7 TB/s).  The card's name, power limit and max SM clock are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lipsync_b200 as lb  # noqa: E402

HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU


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
    ap.add_argument("--windows", type=int, default=64, help="windows re-cropped per call")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--window-s", type=float, default=1.5)
    ap.add_argument("--profile-calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(gpu_info())
    model = lb.LipSyncModel()
    model.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)
    model.to("cuda:0").eval()
    model.compute_precision = "bf16"
    p = lb.Predictor(model, batch_size=64)
    T, H, W, stride = 32, 96, 96, 8
    names, mats = p.robustness_variants(T, H, W)
    K = len(names)
    rows = a.windows * K
    n_plain = rows                                                   # the same number of scored windows per call
    n_frames = (n_plain - 1) * stride + T
    g = torch.Generator().manual_seed(0)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    ta_full = int(n_frames * 100 / 25)
    mel = (-80.0 * torch.rand((1, 80, ta_full), generator=g)).cuda()
    plain_starts = [i * stride for i in range(n_plain)]
    warp_starts = plain_starts[:: max(1, n_plain // a.windows)][: a.windows]   # spread over the track
    plain = lambda: p.score_track_logits(track, plain_starts, mel, n_frames)  # noqa: E731
    warp = lambda: p.score_track_warps(track, warp_starts, mel, n_frames, mats)  # noqa: E731
    with torch.no_grad():
        for _ in range(2):
            plain()
            warp()
        torch.cuda.synchronize()
        # the identity column is the plain window: same bits as score_track_logits
        col0 = warp()[:, 0]
        ref = p.score_track_logits(track, warp_starts, mel, n_frames)
        bitwise = bool(torch.equal(col0, ref))
        tp, to = [], []
        for _ in range(a.reps):
            tp.append(time_block(plain, a.window_s))
            to.append(time_block(warp, a.window_s))
        # builder kernel time, in a run of its own
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.profile_calls):
                warp()
            torch.cuda.synchronize()
    kern_us = [ev.device_time_total or ev.time_range.elapsed_us() for ev in prof.events() if "warp_windows_kernel" in ev.name]
    batches = -(-rows // p.batch_size)
    frame_bytes = T * H * W * 3
    res.update({
        "windows": a.windows, "variants": K, "rows_per_call": rows, "plain_windows_per_call": n_plain, "batch": p.batch_size,
        "plain_rows_per_s": round(n_plain / (median(tp) * 1e-3), 1), "warp_rows_per_s": round(rows / (median(to) * 1e-3), 1),
        "plain_ms_all": [round(x, 3) for x in tp], "warp_ms_all": [round(x, 3) for x in to],
        "warp_over_plain": round((rows / median(to)) / (n_plain / median(tp)), 4),
        "identity_bitwise_equal": bitwise,
        "kernel_launches_profiled": len(kern_us), "kernel_batches_expected": batches * a.profile_calls,
    })
    if kern_us:
        per_batch_bytes = 2 * p.batch_size * frame_bytes
        us = median(kern_us)
        res.update({"kernel_us_median": round(us, 2), "kernel_us_all_min_max": [round(min(kern_us), 2), round(max(kern_us), 2)],
                    "kernel_bytes_per_full_batch": per_batch_bytes, "kernel_gb_per_s": round(per_batch_bytes / (us * 1e-6) / 1e9, 1),
                    "kernel_share_of_7_7_tb_s": round(per_batch_bytes / (us * 1e-6) / HBM_BYTES_PER_S, 3)})
    res["timing"] = (f"CUDA events, blocks of >= {a.window_s} s after warm-up, plain / warps alternating, median of {a.reps}; "
                     f"kernel: torch.profiler over {a.profile_calls} calls, median launch (all batches of 64 rows are full)")
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    assert bitwise, "the identity column differs from score_track_logits"


if __name__ == "__main__":
    main()
