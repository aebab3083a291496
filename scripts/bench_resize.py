"""Resolution robustness on one GPU: `Predictor.score_track_resizes` with the K=8 face sizes of `resolution_track` (64 windows x 8 =
512 rows) against `Predictor.score_track_logits` on 512 plain windows of the same uint8 track, bf16 tensor-core route, inputs
resident on the device, batch 64 with the double (pipelined) workspace.  Prints one JSON line (also written to --out).

Timing: CUDA events around blocks of back-to-back calls of >= --window-s seconds after warm-up; the two calls alternate block
by block so both see the same clocks; the median block is reported as rows per second.  The track (4 120 frames, 114 MB)
is close to the 126 MB L2, so part of a window's frames may be served from L2.  The builder kernel (`resize_windows_kernel`) is
then timed on its own: CUDA events around back-to-back `lsd_resize_windows` calls that build one scoring batch (8 windows x the
8 variants = 64 rows, 2 048 frames; each call also makes two small host-to-device copies, its tables and window starts), and,
in a separate torch.profiler pass over scoring calls, the kernel's device time per batch.  The card's name, power limit and max
SM clock are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

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
    ap.add_argument("--windows", type=int, default=64, help="windows resized per call")
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
    names, variants = p.resolution_variants(H, W)
    K = len(names)
    rows = a.windows * K
    n_plain = rows                                                   # the same number of scored windows per call
    n_frames = (n_plain - 1) * stride + T
    g = torch.Generator().manual_seed(0)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    ta_full = int(n_frames * 100 / 25)
    mel = (-80.0 * torch.rand((1, 80, ta_full), generator=g)).cuda()
    plain_starts = [i * stride for i in range(n_plain)]
    rs_starts = plain_starts[:: max(1, n_plain // a.windows)][: a.windows]   # spread over the track
    plain = lambda: p.score_track_logits(track, plain_starts, mel, n_frames)  # noqa: E731
    resize = lambda: p.score_track_resizes(track, rs_starts, mel, n_frames, variants)  # noqa: E731
    # one scoring batch of the builder alone, through the C-ABI with preallocated buffers
    nb_win = p.batch_size // K
    L = _cabi.lib()
    h = model._ensure_handle(model._device())
    vc = (_cabi.LsdResize * K)(*[_cabi.LsdResize(hh, ww) for hh, ww in variants])
    b_starts = (C.c_int32 * nb_win)(*rs_starts[:nb_win])
    b_out = torch.empty((nb_win * K * T, H, W, 3), dtype=torch.uint8, device="cuda")
    b_ws = torch.empty(int(L.lsd_resize_windows_workspace_bytes(nb_win, K, T, H, W)), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def build():
        rc = L.lsd_resize_windows(h.ptr, track.data_ptr(), n_frames, H, W, b_starts, nb_win, T, vc, K, b_out.data_ptr(),
                                  b_ws.data_ptr(), b_ws.numel(), stream)
        _cabi.check(h.ptr, rc)

    with torch.no_grad():
        for _ in range(2):
            plain()
            resize()
            build()
        torch.cuda.synchronize()
        # the plain column is the plain window: same bits as score_track_logits
        col0 = resize()[:, 0]
        ref = p.score_track_logits(track, rs_starts, mel, n_frames)
        bitwise = bool(torch.equal(col0, ref))
        tp, tj, tb = [], [], []
        for _ in range(a.reps):
            tp.append(time_block(plain, a.window_s))
            tj.append(time_block(resize, a.window_s))
            tb.append(time_block(build, a.window_s / 3))
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.profile_calls):
                resize()
            torch.cuda.synchronize()
    kern_us = [ev.device_time_total or ev.time_range.elapsed_us() for ev in prof.events() if "resize_windows_kernel" in ev.name]
    batches = -(-rows // p.batch_size)
    batch_ms = median(tj) / batches
    res.update({
        "windows": a.windows, "variants": K, "variant_names": names, "rows_per_call": rows, "plain_windows_per_call": n_plain,
        "batch": p.batch_size,
        "plain_rows_per_s": round(n_plain / (median(tp) * 1e-3), 1), "resize_rows_per_s": round(rows / (median(tj) * 1e-3), 1),
        "plain_ms_all": [round(x, 3) for x in tp], "resize_ms_all": [round(x, 3) for x in tj],
        "resize_over_plain": round((rows / median(tj)) / (n_plain / median(tp)), 4),
        "plain_column_bitwise_equal": bitwise,
        "builder_call_us_events": round(median(tb) * 1e3, 2), "builder_call_us_all": [round(x * 1e3, 2) for x in tb],
        "builder_rows_per_call": nb_win * K, "builder_share_of_scoring_batch": round(median(tb) / batch_ms, 4),
        "kernel_launches_profiled": len(kern_us), "kernel_batches_expected": batches * a.profile_calls,
    })
    if kern_us:
        res.update({"kernel_us_median_profiler": round(median(kern_us), 2),
                    "kernel_us_all_min_max_profiler": [round(min(kern_us), 2), round(max(kern_us), 2)]})
    res["timing"] = (f"CUDA events, blocks of >= {a.window_s} s after warm-up, plain / resize / builder alternating, median of {a.reps}; "
                     f"builder: lsd_resize_windows of one 64-row batch; kernel: torch.profiler over {a.profile_calls} scoring calls, "
                     f"median launch (all batches of 64 rows are full)")
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    assert bitwise, "the plain column differs from score_track_logits"


if __name__ == "__main__":
    main()
