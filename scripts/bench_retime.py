"""Temporal robustness on one GPU: `Predictor.score_track_retimes` with the K=12 default retime variants of `temporal_track` at
15 fps (64 windows x 12 = 768 rows) against `Predictor.score_track_logits` on 768 plain windows of the same uint8 track, bf16
tensor-core route, inputs resident on the device, batch 64 with the double (pipelined) workspace.  Prints one JSON line (also
written to --out).

Timing: CUDA events around blocks of back-to-back calls of >= --window-s seconds after warm-up; the calls alternate block by
block so all see the same clocks; the median block is reported.  The track (6 168 frames, 171 MB) is larger than the 126 MB L2.
The builder kernel (`retime_windows_kernel`) is timed on its own: CUDA events around back-to-back `lsd_retime_windows` calls that
build all 768 rows (24 576 frames, 680 MB written; each call also makes two small host-to-device copies, its tables and window
starts), reported per 64-row scoring batch (the call's time / 12).  Its bytes are those the tables imply: every output frame is
written once and every tap of nonzero weight reads one frame (frames shared by the variants of a window are counted once per
tap, so part of these reads is served from L2).  A separate torch.profiler pass over scoring calls gives the kernel's device time
per scoring batch.  The card's name, power limit and max SM clock are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lipsync_b200 as lb  # noqa: E402
from lipsync_b200 import _cabi  # noqa: E402


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
    ap.add_argument("--windows", type=int, default=64, help="windows retimed per call")
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
    names, tabs, _ = p.temporal_variants(T, 15.0)
    K = len(names)
    rows = a.windows * K
    n_plain = rows                                                   # the same number of scored windows per call
    n_frames = (n_plain - 1) * stride + T
    g = torch.Generator().manual_seed(0)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    ta_full = int(n_frames * 100 / 25)
    mel = (-80.0 * torch.rand((1, 80, ta_full), generator=g)).cuda()
    plain_starts = [i * stride for i in range(n_plain)]
    rt_starts = plain_starts[:: max(1, n_plain // a.windows)][: a.windows]   # spread over the track
    plain = lambda: p.score_track_logits(track, plain_starts, mel, n_frames)  # noqa: E731
    retime = lambda: p.score_track_retimes(track, rt_starts, mel, n_frames, tabs)  # noqa: E731
    # the builder alone over all rows, through the C-ABI with preallocated buffers
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    _, vc = p._retime_args(track, rt_starts, tabs)
    b_starts = (C.c_int32 * a.windows)(*rt_starts)
    b_out = torch.empty((rows * T, H, W, 3), dtype=torch.uint8, device="cuda")
    b_ws = torch.empty(int(L.lsd_retime_windows_workspace_bytes(a.windows, K, T, H, W)), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    fb = H * W * 3
    taps = sum(int((np.asarray(w) > 0).sum()) for _, w in tabs)       # nonzero taps over the K*T output frames of one window
    builder_bytes = a.windows * (K * T + taps) * fb

    def build():
        rc = L.lsd_retime_windows(h.ptr, track.data_ptr(), n_frames, H, W, b_starts, a.windows, T, vc, K, b_out.data_ptr(),
                                  b_ws.data_ptr(), b_ws.numel(), stream)
        _cabi.check(h.ptr, rc)

    with torch.no_grad():
        for _ in range(2):
            plain()
            retime()
            build()
        torch.cuda.synchronize()
        # the `none` column is the plain window: same bits as score_track_logits
        col0 = retime()[:, 0]
        ref = p.score_track_logits(track, rt_starts, mel, n_frames)
        bitwise = bool(torch.equal(col0, ref))
        tp, tr, tb = [], [], []
        for _ in range(a.reps):
            tp.append(time_block(plain, a.window_s))
            tr.append(time_block(retime, a.window_s))
            tb.append(time_block(build, a.window_s / 3))
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.profile_calls):
                retime()
            torch.cuda.synchronize()
    kern_us = [ev.device_time_total or ev.time_range.elapsed_us() for ev in prof.events() if "retime_windows_kernel" in ev.name]
    batches = -(-rows // p.batch_size)
    batch_ms = median(tr) / batches
    per_batch_us = median(tb) * 1e3 / batches
    res.update({
        "windows": a.windows, "variants": K, "variant_names": names, "rows_per_call": rows, "plain_windows_per_call": n_plain,
        "batch": p.batch_size,
        "plain_rows_per_s": round(n_plain / (median(tp) * 1e-3), 1), "retime_rows_per_s": round(rows / (median(tr) * 1e-3), 1),
        "plain_ms_all": [round(x, 3) for x in tp], "retime_ms_all": [round(x, 3) for x in tr],
        "retime_over_plain": round((rows / median(tr)) / (n_plain / median(tp)), 4),
        "none_column_bitwise_equal": bitwise,
        "builder_call_rows": rows, "builder_call_us_events": round(median(tb) * 1e3, 2),
        "builder_call_us_all": [round(x * 1e3, 2) for x in tb],
        "builder_us_per_64_row_batch": round(per_batch_us, 2), "builder_share_of_scoring_batch": round(per_batch_us * 1e-3 / batch_ms, 4),
        "builder_table_bytes_per_call": builder_bytes, "builder_table_gb_per_s": round(builder_bytes / (median(tb) * 1e-3) / 1e9, 1),
        "kernel_launches_profiled": len(kern_us), "kernel_batches_expected": batches * a.profile_calls,
    })
    if kern_us:
        res.update({"kernel_us_median_profiler": round(median(kern_us), 2),
                    "kernel_us_all_min_max_profiler": [round(min(kern_us), 2), round(max(kern_us), 2)]})
    res["timing"] = (f"CUDA events, blocks of >= {a.window_s} s after warm-up, plain / retime / builder alternating, median of {a.reps}; "
                     f"builder: lsd_retime_windows of all {rows} rows, per 64-row batch = call / {batches}; kernel: torch.profiler "
                     f"over {a.profile_calls} scoring calls, median launch (all batches of 64 rows are full)")
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    assert bitwise, "the none column differs from score_track_logits"


if __name__ == "__main__":
    main()
