#!/usr/bin/env python
"""Benchmark of the window-scoring hot path (BASELINE.json: windows/sec at 1/2/4/8 B200 + roofline fraction,
next to the reference's CPU path timed on the box's own host cores).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one JSON line on rank 0)
  python bench.py --impl reference --gpus N ...             # the reference algorithm on the host cores (oracle port)
  python bench.py ... --dump-outputs DIR                    # also write the last timed step's logits of every path as DIR/*.npy

A "step" is one pass of the hot path over one batch of B=64 synthetic canonical windows per GPU
(video (64,3,32,96,96) + log-mel (64,1,80,128); BASELINE.json configs[1]).  `value` is timed with the inputs already
resident in HBM; `e2e` is the same metric through the public API with pinned HOST buffers (H2D of the windows and
D2H of the logits inside the timed region).  Weak scaling: every rank scores its own batch; under N>1 the per-step
logits are all-gathered (NCCL) as in the long-video path (the only collective on the path).
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_WINDOW = 31.29e9   # SURVEY.md §2.3 / §8d: 2*MACs of LipSyncModel.forward at the canonical window
BATCH = 64
WORKLOAD = "batched window scoring B=64 per GPU, canonical window video(3,32,96,96)+logmel(1,80,128), random-init R2Plus1D-Sync"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def _dist():
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return ws, rank, local


CPU_SWEEP = (1, 4, 8, 16)


def cpu_reference_sweep(steps: int, warmup: int, batches=CPU_SWEEP):
    """The reference algorithm (oracle port of LipSyncModel.forward, fp32, torch CPU, all host threads) per BASELINE.md §4:
    `warmup` untimed + `steps` timed forwards at every B of the sweep; per B the best and the median time; the reported
    throughput is the best over B of B / best_time (the most favourable figure for the baseline)."""
    import lipsync_b200 as lb
    from oracle import lipsync_oracle as orc
    torch.set_num_threads(os.cpu_count() or 1)
    sd = lb.make_synthetic_state_dict(0)
    video, audio = lb.synthetic_windows(1, max(batches))
    per_b = {}
    for b in batches:
        v, a = video[:b], audio[:b]
        for _ in range(warmup):
            orc.forward(sd, v, a)
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            orc.forward(sd, v, a)
            ts.append(time.perf_counter() - t0)
        ts.sort()
        per_b[b] = {"best_ms": ts[0] * 1e3, "median_ms": ts[len(ts) // 2] * 1e3,
                    "windows_per_s_best": b / ts[0], "windows_per_s_median": b / ts[len(ts) // 2]}
    best_b = max(per_b, key=lambda b: per_b[b]["windows_per_s_best"])
    return per_b, best_b, torch.get_num_threads()


def _cpu_baseline_record(per_b, best_b, cores, steps, warmup):
    r = per_b[best_b]
    return {"value": r["windows_per_s_best"], "unit": "windows/s", "cores": cores, "kind": "port",
            "median_value": r["windows_per_s_median"], "best_batch": best_b,
            "single_window_ms_best": per_b[min(per_b)]["best_ms"], "single_window_ms_median": per_b[min(per_b)]["median_ms"],
            "per_batch": {str(b): v for b, v in per_b.items()},
            "sample": (f"{warmup} warm-up + {steps} timed forwards at each B in {list(per_b)} (canonical windows, fp32, torch CPU, "
                       f"{cores} threads) through the CPU restatement of LipSyncModel.forward (oracle/, pinned on the real reference's "
                       "goldens; /root/reference does not exist on the GPU box); value = best B / best time")}


def run_reference(args, out=sys.stdout):
    ws, rank, _ = _dist()
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    per_b, best_b, cores = cpu_reference_sweep(steps, warmup)
    rec = _cpu_baseline_record(per_b, best_b, cores, steps, warmup)
    line = {
        "impl": "reference", "metric": "windows_per_sec", "value": rec["value"], "unit": "windows/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": per_b[best_b]["best_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_batch": best_b,
                   "note": ("a step of this arm is ONE forward over a bounded sample of the workload (B in {1,4,8,16} canonical windows, the "
                            "best B is reported), not the 64-window batch: the reference is pure Python/PyTorch and is timed through the "
                            "CPU restatement of LipSyncModel.forward on all host threads")},
        "cpu_baseline": rec,
        "e2e": {"value": rec["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=out, flush=True)


def eager_gpu_run(dev, batch: int, steps: int, warmup: int):
    """PyTorch eager on the same B200 (cuDNN / cuBLAS under bf16 autocast, channels_last_3d video): the only other GPU
    implementation of this model (BASELINE.md §4).  A stated baseline: the same restated forward the CPU arm runs, moved to
    the GPU — not part of the product path."""
    import lipsync_b200 as lb
    from oracle import lipsync_oracle as orc
    sd = {k: (v.to(dev).contiguous(memory_format=torch.channels_last_3d) if v.dim() == 5 else v.to(dev))
          for k, v in lb.make_synthetic_state_dict(0).items()}
    v, a = lb.synthetic_windows(1, 4)
    v = v.repeat(batch // 4 + 1, 1, 1, 1, 1)[:batch].to(dev).contiguous(memory_format=torch.channels_last_3d)
    a = a.repeat(batch // 4 + 1, 1, 1, 1)[:batch].to(dev)
    res = {}
    for name, ctx in (("bf16_autocast", lambda: torch.autocast("cuda", dtype=torch.bfloat16)),
                      ("fp16_autocast", lambda: torch.autocast("cuda", dtype=torch.float16))):
        try:
            with torch.no_grad(), ctx():
                for _ in range(warmup):
                    orc.forward(sd, v, a)
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    orc.forward(sd, v, a)
                e1.record()
                torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / steps
            res[name] = {"windows_per_s": batch / ms * 1e3, "ms_per_step": ms}
        except Exception as exc:  # noqa: BLE001  (a baseline leg must never take the bench line down)
            res[name] = {"error": f"{type(exc).__name__}: {str(exc)[:160]}"}
    res["what"] = (f"torch {torch.__version__} eager, cuDNN/cuBLAS, B={batch}, inputs resident, {steps} steps after {warmup} warm-ups; "
                   "same weights and inputs as the main arm")
    return res


def latency_probe(pred, lb, iters: int = 30):
    """Wall-clock latency of the reference-shaped single-window calls (host numpy in, python float out; every call includes
    its H2D copy and the D2H read of the result): `_infer_confidence` (predictor.py:212-244, B=1) and
    `_temporal_smoothed_confidence` (predictor.py:295-331: one full window + three half windows)."""
    import numpy as np
    v, a = lb.synthetic_windows(7, 1)
    v, a = v[0].numpy(), a[0].numpy()
    out = {}
    for name, fn in (("infer_confidence_ms", lambda: pred._infer_confidence(v, a)),
                     ("temporal_smoothed_confidence_ms", lambda: pred._temporal_smoothed_confidence(v, a))):
        for _ in range(5):
            fn()
        ts = []
        for _ in range(iters):
            t0 = time.perf_counter()
            fn()
            ts.append((time.perf_counter() - t0) * 1e3)
        ts.sort()
        out[name] = {"best": ts[0], "median": ts[len(ts) // 2]}
    out["graphs"] = bool(getattr(pred, "use_cuda_graphs", False))
    out["graph_captures"] = int(getattr(pred, "graph_captures", 0))
    out["what"] = "wall clock around the public call on host numpy inputs, B=1 (and 1+3 windows), after 5 warm-ups"
    return out


def long_video_probe(pred, lb, ws, rank, dev, n_windows: int):
    """BASELINE.json configs[4]: `n_windows` sliding windows (stride 8) of ONE synthetic uint8 track, contiguous block partition
    over the ranks (strong scaling), windows built on the device, one all-gather of the fp32 logits, SHA-256 of the gathered
    logits (identical across shardings).  The track is resident in HBM (rank-local span)."""
    import hashlib
    import torch.distributed as dist
    stride, T = 8, 32
    n_frames = stride * (n_windows - 1) + T + 16
    lo, hi = lb.partition_windows(n_windows, ws, rank)
    f_lo, f_hi = stride * lo, stride * max(hi - 1, lo) + T
    g = torch.Generator(device=dev).manual_seed(5)
    track = torch.empty(f_hi - f_lo, 96, 96, 3, dtype=torch.uint8, device=dev)
    blk = 4096
    for f0 in range(0, n_frames, blk):          # same random stream on every rank -> identical track across shardings
        chunk = torch.randint(0, 256, (min(blk, n_frames - f0), 96, 96, 3), dtype=torch.uint8, device=dev, generator=g)
        a, b = max(f0, f_lo), min(f0 + chunk.shape[0], f_hi)
        if b > a:
            track[a - f_lo:b - f_lo] = chunk[a - f0:b - f0]
    del chunk
    ta_full = int(n_frames / 15 * 100)
    gm = torch.Generator().manual_seed(6)
    mel = (-80.0 * torch.rand(1, 80, ta_full, generator=gm)).to(dev)
    starts_abs = [stride * i for i in range(lo, hi)]

    def score_range(_lo, _hi):
        return pred.score_track_logits(track, [s - f_lo for s in starts_abs], mel, n_frames, audio_starts_from=starts_abs)

    def run():
        return pred.score_windows_sharded(n_windows, score_range, ws, rank)

    run()
    torch.cuda.synchronize(dev)
    if ws > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    logits = run()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if ws > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    lg = logits.cpu()
    del track
    rec = {"windows": n_windows, "n_gpus": ws, "scaling": "strong", "ms": ms, "windows_per_s": n_windows / ms * 1e3,
           "logits_sha256_16": hashlib.sha256(lg.numpy().tobytes()).hexdigest()[:16], "fake_votes": int((lg < 0).sum()),
           "what": "uint8 track resident in HBM (rank-local span), windows built on the device, batches pipelined, one all-gather of fp32 logits"}
    return rec, lg


DUMP_MAX_ELEMS = 4 << 20     # 16 MB of float32 per array: the dump of a run stays below 64 MB in all


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each flattened array as `out_dir/<name>.npy` in float32.  An array longer than DUMP_MAX_ELEMS (only config5's
    logits, at a large --config5-windows) is stored as every k-th element, the smallest k that fits: a fixed sample, so two
    runs with the same arguments store the same windows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().to("cpu", torch.float32).reshape(-1)
        a = a[::-(-a.numel() // DUMP_MAX_ELEMS)] if a.numel() > DUMP_MAX_ELEMS else a
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def _claim_stdout():
    """Keep a private handle on the real stdout for the single JSON line and point fd 1 at stderr: libraries (NCCL's version
    banner, nvcc through build()) write to fd 1 behind Python's back."""
    real = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    return real


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-gpu", action="store_true")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--config5-windows", type=int, default=10000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the logits each timed path returned in its last step as DIR/<name>.npy "
                         "(float32; rank 0) so that two builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
        return run_reference(args, out)

    import __graft_entry__ as ge
    ws, rank, local = _dist()
    if rank == 0:
        ge.build()
    import torch.distributed as dist
    if ws > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    ge.build()
    import lipsync_b200 as lb

    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    B, K, W = args.batch, args.steps, max(3, args.warmup)
    model = lb.LipSyncModel()
    model.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)
    model.to(dev).eval()
    model.compute_precision = args.precision
    pred = lb.Predictor(model, batch_size=B)

    # synthetic inputs (host, pinned) and their device-resident copies; distinct data per rank
    # (video values are k/255 for integer k, exactly what the reference's window builder produces from uint8 mouth crops:
    #  astype(float32) / 255.0, video.py:552-556 — timing does not depend on the values, the e2e transport does)
    _, ah = lb.synthetic_windows(100 + rank, 4)
    gv = torch.Generator().manual_seed(100 + rank)
    vh = torch.randint(0, 256, (4, 3, 32, 96, 96), dtype=torch.uint8, generator=gv).to(torch.float32) / 255.0
    vh = vh.repeat(B // 4 + 1, 1, 1, 1, 1)[:B].contiguous().pin_memory()
    ah = ah.repeat(B // 4 + 1, 1, 1, 1)[:B].contiguous().pin_memory()
    vd, ad = vh.to(dev), ah.to(dev)
    # N > 1: every rank keeps the logits of its K batches and ONE all-gather at the end of the timed region hands all of them
    # to every rank — the path's only exchange step (long videos gather per-window logits once, before the aggregation)
    local_logits = torch.empty(max(K, W), B, dtype=torch.float32, device=dev)
    gathered = torch.empty(ws * max(K, W) * B, dtype=torch.float32, device=dev) if ws > 1 else None
    gathered_e2e = torch.empty(ws * B, dtype=torch.float32, device=dev) if ws > 1 else None
    step_no = [0]

    def step_resident():
        logits = model(vd, ad)
        if ws > 1:
            local_logits[step_no[0] % local_logits.shape[0]].copy_(logits)
            step_no[0] += 1
        return logits

    def gather_resident():
        if ws > 1:
            dist.all_gather_into_tensor(gathered, local_logits.view(-1))

    e2e_h2d_bytes, e2e_transport = [0], ["fp32"]

    pred_f32 = lb.Predictor(model, batch_size=B, host_transport="fp32")

    def run_e2e(steps, p=None):
        """Public API on HOST buffers: Predictor.score_batches uploads every step's windows from pinned host memory
        (copy stream, overlapped with the previous step's scoring) and reads every step's logits back."""
        p = pred if p is None else p
        outs = p.score_batches((vh, ah) for _ in range(steps))
        if p is pred:
            e2e_h2d_bytes[0] = int(p.last_h2d_bytes_per_batch)
            e2e_transport[0] = p.last_transport
        if ws > 1:
            last = outs[-1].to(dev)
            dist.all_gather_into_tensor(gathered_e2e, last)
            return gathered_e2e.cpu()
        return outs[-1]

    def timed(fn, steps, profile=False, whole=False, finalize=None):
        if whole:
            fn(W)
        else:
            for _ in range(W):
                fn()
        if finalize is not None:
            finalize()
        torch.cuda.synchronize(dev)
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        sampler = ClockSampler(local)
        sampler.start()
        if profile:
            model.profile_enable(2 if args.precision == 'bf16' else 1)
        n0 = model.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        last = None
        e0.record()
        if whole:
            last = fn(steps)
        else:
            for _ in range(steps):
                last = fn()
        if finalize is not None:
            finalize()
        e1.record()
        torch.cuda.synchronize(dev)
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        launches = model.launch_count() - n0
        prof = model.profile_get() if profile else None
        if profile:
            model.profile_enable(False)
        sampler.stop_flag = True
        sampler.join()
        if ws > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, prof, sampler.result(), last

    # uint8-track variant of the end-to-end path (SURVEY.md §8f-1): per step the host hands over the uint8 mouth-crop span of
    # the step's 64 windows (stride 8: 536 frames, 14.8 MB instead of 226 MB of fp32 windows) from pinned memory, the windows
    # are built on the device (lsd_score_windows), and the logits come back to the host.
    n_tf = 8 * (B - 1) + 32
    gt = torch.Generator().manual_seed(200 + rank)
    track_h = torch.randint(0, 256, (n_tf, 96, 96, 3), dtype=torch.uint8, generator=gt).pin_memory()
    mel_h = (-80.0 * torch.rand(1, 80, int(n_tf / 15 * 100), generator=gt)).pin_memory()
    starts = [8 * i for i in range(B)]
    track_slots = [torch.empty_like(track_h, device=dev) for _ in range(2)]
    mel_slots = [torch.empty_like(mel_h, device=dev) for _ in range(2)]
    copy_stream = torch.cuda.Stream(dev)

    def run_e2e_track(steps):
        comp = torch.cuda.current_stream(dev)
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        free = [torch.cuda.Event(), torch.cuda.Event()]
        for e in free:
            e.record(comp)
        host_out = []
        for k in range(steps):
            sl = k & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(free[sl])
                track_slots[sl].copy_(track_h, non_blocking=True)
                mel_slots[sl].copy_(mel_h, non_blocking=True)
                ready[sl].record(copy_stream)
            comp.wait_event(ready[sl])
            lg = pred.score_track_logits(track_slots[sl], starts, mel_slots[sl], n_tf)
            free[sl].record(comp)
            ho = torch.empty(B, dtype=torch.float32, pin_memory=True)
            ho.copy_(lg, non_blocking=True)
            host_out.append(ho)
        comp.synchronize()
        return host_out[-1]

    # outputs of the last timed step of every path (the `value`, `e2e*` and `config5` figures), for --dump-outputs
    last_out = {}
    ms, launches, prof, clocks, last_out["logits"] = timed(step_resident, K, profile=True, finalize=gather_resident)
    if ws > 1:      # what every rank receives for the last step: the logits of all ranks
        rows = local_logits.shape[0]
        last_out["logits"] = gathered.view(ws, rows, B)[:, (step_no[0] - 1) % rows].clone()
    ms_e2e, _, _, _, last_out["e2e_logits"] = timed(run_e2e, K, whole=True)
    ms_e2e_f32, _, _, _, last_out["e2e_fp32_upload_logits"] = timed(lambda n: run_e2e(n, pred_f32), K, whole=True)
    ms_trk, _, _, _, last_out["e2e_track_u8_logits"] = timed(run_e2e_track, K, whole=True)
    # sustained: the same resident step back to back for >= ~1.5 s (the K-step region above lasts ~60 ms: a burst figure, taken
    # before the 1000 W power cap pulls the SM clock down)
    k_sus = max(K, int(1500.0 / max(ms / K, 0.05)))
    if ws > 1:
        local_logits = torch.empty(1, B, dtype=torch.float32, device=dev)     # (the sustained run keeps only the last batch)
    ms_sus, _, _, clocks_sus, _ = timed(step_resident, k_sus)
    value = ws * B * K / (ms / 1e3)
    e2e = ws * B * K / (ms_e2e / 1e3)
    e2e_trk = ws * B * K / (ms_trk / 1e3)

    # latency of the reference-shaped single-window calls (predictor.py:212-244, 295-331): host numpy in, python float out
    lat = None
    if args.precision == "bf16":
        lat = latency_probe(pred, lb)
    # BASELINE.json configs[4]: 10 000 sliding windows of one uint8 track, sharded over the ranks (strong scaling)
    c5 = None
    if not args.no_config5:
        c5, last_out["config5_logits"] = long_video_probe(pred, lb, ws, rank, dev, args.config5_windows)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_out)

    if rank == 0:
        peaks, peak_src = _peaks()
        kern_ms, kern_n, kern_flops = prof
        # dominant kernel class: the implicit-GEMM convolution/linear kernel (tensor-bound on the bf16 path)
        achieved = (kern_flops / max(kern_n, 1)) / ((kern_ms / max(kern_n, 1)) * 1e-3) / 1e12 if kern_n else 0.0
        peak = float(peaks.get("bf16_tflops", 1590.0))                       # burst: the timed region lasts ~60 ms at full clocks
        peak_sus = float(peaks.get("bf16_tflops_sustained", peak))
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            with open(tp) as fh:
                traffic = json.load(fh).get("dram_bytes_per_launch")
        line = {
            "metric": "windows_per_sec", "value": value, "unit": "windows/s", "n_gpus": ws, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "precision": args.precision,
                       "l2": "inputs (226 MB fp32 video per step) exceed the 126 MB L2; no explicit flush",
                       "timed_region": f"{K} steps = {ms:.0f} ms: burst conditions (see `sustained` for >= 1.5 s back to back)",
                       "parallelism": f"dp{ws} (independent windows; all-gather of fp32 logits only)"},
            "gpu_launches": launches,
            "clocks": clocks,
            "sustained": {"value": ws * B * k_sus / (ms_sus / 1e3), "unit": "windows/s", "steps": k_sus, "ms_per_step": ms_sus / k_sus,
                          "seconds": ms_sus / 1e3, "clocks": clocks_sus},
            "e2e": {"value": e2e, "unit": "windows/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": e2e_h2d_bytes[0], "d2h_bytes_per_step": (ws if ws > 1 else 1) * B * 4,
                    "api": ("Predictor.score_batches on pinned host fp32 windows (per step: exact-uint8 detection + packing on the host "
                            "threads when the windows are u8/255 as video.py:552-556 produces them, H2D on a copy stream, forward, D2H "
                            "of the logits)"),
                    "transport": e2e_transport[0], "host_pack_threads": pred.host_pack_threads},
            "e2e_fp32_upload": {"value": ws * B * K / (ms_e2e_f32 / 1e3), "unit": "windows/s", "ms_per_step": ms_e2e_f32 / K,
                                "h2d_bytes_per_step": vh.numel() * 4 + ah.numel() * 4, "d2h_bytes_per_step": (ws if ws > 1 else 1) * B * 4,
                                "api": "the same call with host_transport='fp32' (windows cross PCIe as fp32: round 1's e2e)"},
            "e2e_track_u8": {"value": e2e_trk, "unit": "windows/s", "ms_per_step": ms_trk / K,
                             "h2d_bytes_per_step": track_h.numel() + mel_h.numel() * 4, "d2h_bytes_per_step": B * 4,
                             "api": "Predictor.score_track_logits on a pinned host uint8 mouth-crop track (windows built on the device, lsd_score_windows)"},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "peak_sustained": peak_sus, "frac_of_sustained": achieved / peak_sus,
                         "traffic": traffic,
                         "traffic_source": "static: per-launch dram__bytes_read+write from the committed ncu --set full capture (profiles/traffic.json), not measured in this run",
                         "peak_source": f"{peak_src} bf16_tflops (burst: kernels timed in a {ms:.0f} ms region at full clocks)",
                         "kernel": ("stem_ring_kernel + umma_conv_kernel, the 9 tcgen05 launches of the 3-D conv visual encoder (stem + layer1-4: 26.77 of the 31.29 "
                                    "GFLOP per window); CUDA events on the launch stream"
                                    if args.precision == "bf16" else "conv_f32_kernel (all launches, CUDA events on the launch stream)"),
                         "kernel_ms_per_step": kern_ms / K, "kernel_launches_per_step": kern_n / K,
                         "kernel_share_of_step": kern_ms / ms,
                         "whole_model_tflops": FLOP_PER_WINDOW * B * K / (ms / 1e3) / 1e12,
                         "whole_model_frac": FLOP_PER_WINDOW * B * K / (ms / 1e3) / 1e12 / peak},
        }
        if lat is not None:
            line["latency"] = lat
        if c5 is not None:
            line["config5"] = c5
        if ws == 1 and not args.no_cpu_baseline:
            per_b, best_b, cores = cpu_reference_sweep(10, 3)
            line["cpu_baseline"] = _cpu_baseline_record(per_b, best_b, cores, 10, 3)
        if ws == 1 and not args.no_eager_gpu and args.precision == "bf16":
            line["eager_gpu"] = eager_gpu_run(dev, B, 5, 3)
        print(json.dumps(line), file=out, flush=True)
    if ws > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
