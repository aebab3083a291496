"""Audio occlusion evidence on one GPU: `Predictor.score_track_audio_occlusions` (64 windows x K=17 boxes = 1088 rows) against
(1) the same 1088 masked rows scored by the plain path: the masked log-mel slices built once on the host and laid end to end as
one clip, each window's start repeated K times, `lsd_score_windows` with explicit audio starts r*Ta and the double (pipelined)
workspace; (2) `Predictor.score_track_occlusions` with its default 25 boxes on the same 64 windows (1600 rows), per row.
bf16 tensor-core route, inputs resident on the device, batch 64.  Prints one JSON line (also written to --out).

Timing: CUDA events around blocks of back-to-back calls of >= --window-s seconds after warm-up; the three calls alternate block
by block so all see the same clocks; the median block is reported as rows per second.  The track (8 728 frames, 241 MB) exceeds
the 126 MB L2.  A separate torch.profiler pass times the builder kernel (`mask_audio_windows_kernel`) and sets it against the
bytes it writes, F x rows x Ta x 4 per batch, over the HBM bandwidth of the data sheet (7.7 TB/s); its reads are the 64 windows'
slices, mostly served from L2.  The card's name, power limit and max SM clock are read in the same run."""
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


def plain_rows(p, track, starts, clip, total_v_frames, Ta):
    """lsd_score_windows over `starts` with explicit audio starts r*Ta into `clip`, in a double workspace (returns a callable)."""
    m = p.model
    n = len(starts)
    H, W, F, Ta_full = int(track.shape[1]), int(track.shape[2]), int(clip.shape[1]), int(clip.shape[2])
    L = _cabi.lib()
    h = m._ensure_handle(m._device())
    prec = m._precision()
    batch = min(p.batch_size, n)
    need = L.lsd_score_workspace_bytes(h.ptr, batch, p.chunk_size, H, W, F, Ta, prec)
    ws = torch.empty(2 * need, dtype=torch.uint8, device="cuda")
    out = torch.empty(n, dtype=torch.float32, device="cuda")
    st = (C.c_int32 * n)(*starts)
    ast = (C.c_int32 * n)(*[r * Ta for r in range(n)])

    def run():
        with m._lsd_lock:
            rc = L.lsd_score_windows(h.ptr, track.data_ptr(), int(track.shape[0]), H, W, st, ast, n, p.chunk_size, clip.data_ptr(), F,
                                     Ta_full, total_v_frames, Ta, prec, batch, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                     torch.cuda.current_stream().cuda_stream)
            _cabi.check(h.ptr, rc)
        return out
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=64, help="windows explained per call")
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
    T, H, W, F, Ta, stride, fill = 32, 96, 96, 80, 128, 8, -80.0
    boxes = [(0, 0, 0, 0)] + p.mute_segment_boxes(Ta, 16, F) + p.mel_band_boxes(Ta, F, 8)
    vboxes = [(0, 0, 0, 0, 0, 0, -1)] + p.freeze_segment_boxes(T, 4, H, W) + p.fill_cell_boxes(T, H, W, 4)
    K, KV = len(boxes), len(vboxes)
    rows, vrows = a.windows * K, a.windows * KV
    n_track = rows                                                   # the track of bench_occlusion.py at 1088 windows
    n_frames = (n_track - 1) * stride + T
    g = torch.Generator().manual_seed(0)
    track = torch.randint(0, 256, (n_frames, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    ta_full = int(n_frames * 100 / 25)
    mel = (-80.0 * torch.rand((1, F, ta_full), generator=g)).cuda()
    all_starts = [i * stride for i in range(n_track)]
    starts = all_starts[:: max(1, n_track // a.windows)][: a.windows]  # spread over the track
    # the reference construction: masked slices on the host, end to end as one clip
    host = mel.cpu().numpy()
    slices = []
    for s in starts:
        win = p._align_audio_chunk(host, s, n_frames, Ta)[0]
        for c0, c1, f0, f1 in boxes:
            w = win.copy()
            w[f0:f1, c0:c1] = fill
            slices.append(w)
    clip = torch.from_numpy(np.concatenate(slices, axis=1)[None]).cuda()
    rep_starts = [s for s in starts for _ in boxes]
    aud = lambda: p.score_track_audio_occlusions(track, starts, mel, n_frames, boxes, fill=fill)  # noqa: E731
    plain = plain_rows(p, track, rep_starts, clip, n_frames, Ta)
    vis = lambda: p.score_track_occlusions(track, starts, mel, n_frames, vboxes)  # noqa: E731
    with torch.no_grad():
        for _ in range(2):
            aud()
            plain()
            vis()
        torch.cuda.synchronize()
        out = aud().clone()
        ref = p.score_track_logits(track, starts, mel, n_frames)
        bitwise = bool(torch.equal(out[:, 0], ref))                  # the empty box is the plain window
        plain_bitwise = bool(torch.equal(out.flatten(), plain()))    # every row is the plain path's row
        ta, tp, tv = [], [], []
        for _ in range(a.reps):
            ta.append(time_block(aud, a.window_s))
            tp.append(time_block(plain, a.window_s))
            tv.append(time_block(vis, a.window_s))
        # builder kernel time, in a run of its own
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.profile_calls):
                aud()
            torch.cuda.synchronize()
    kern_us = [ev.device_time_total or ev.time_range.elapsed_us() for ev in prof.events() if "mask_audio_windows_kernel" in ev.name]
    batches = -(-a.windows // p.batch_size)
    aud_rps, plain_rps, vis_rps = rows / (median(ta) * 1e-3), rows / (median(tp) * 1e-3), vrows / (median(tv) * 1e-3)
    res.update({
        "windows": a.windows, "boxes": K, "rows_per_call": rows, "batch_windows": p.batch_size, "fill": fill,
        "audio_occlusion_ms_per_call": round(median(ta), 3), "audio_occlusion_rows_per_s": round(aud_rps, 1),
        "plain_rows_per_s": round(plain_rps, 1), "audio_over_plain_per_row": round(aud_rps / plain_rps, 3),
        "visual_occlusion_boxes": KV, "visual_occlusion_rows_per_call": vrows, "visual_occlusion_rows_per_s": round(vis_rps, 1),
        "audio_over_visual_occlusion_per_row": round(aud_rps / vis_rps, 3),
        "audio_occlusion_ms_all": [round(x, 3) for x in ta], "plain_ms_all": [round(x, 3) for x in tp],
        "visual_occlusion_ms_all": [round(x, 3) for x in tv],
        "empty_box_bitwise_equal": bitwise, "plain_path_bitwise_equal": plain_bitwise,
        "kernel_launches_profiled": len(kern_us), "kernel_batches_expected": batches * a.profile_calls,
    })
    if kern_us:
        written = F * p.batch_size * K * Ta * 4
        us = median(kern_us)
        res.update({"kernel_us_median": round(us, 2), "kernel_us_all_min_max": [round(min(kern_us), 2), round(max(kern_us), 2)],
                    "kernel_bytes_written_per_full_batch": written, "kernel_write_gb_per_s": round(written / (us * 1e-6) / 1e9, 1),
                    "kernel_write_share_of_7_7_tb_s": round(written / (us * 1e-6) / HBM_BYTES_PER_S, 3)})
    res["timing"] = (f"CUDA events, blocks of >= {a.window_s} s after warm-up, audio occlusion / plain rows / visual occlusion "
                     f"alternating, median of {a.reps}; kernel: torch.profiler over {a.profile_calls} calls, median launch")
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    assert bitwise, "the empty-box column differs from score_track_logits"
    assert plain_bitwise, "audio occlusion rows differ from the plain path on the host-masked clip"


if __name__ == "__main__":
    main()
