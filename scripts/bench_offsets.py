"""Audio-offset sweep on one GPU: `LipSyncModel.forward_audio_variants` (visual side once, K audio windows per video) against
K plain forwards with the shifted audio, and one plain B=64 forward, all resident, bf16 tensor-core route.  Prints one JSON line
(also written to --out).  Timing: CUDA events around blocks of back-to-back calls of >= --window-s seconds after warm-up; the
shared and the naive route alternate block by block so both see the same clocks; the median block is reported.  The inputs
(226 MB of video for 64 windows) exceed the 126 MB L2.  The script checks that shared and naive logits are bit-identical."""
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
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--ks", default="1,7,15")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--window-s", type=float, default=1.5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    B = a.batch
    ks = [int(k) for k in a.ks.split(",")]
    res = dict(gpu_info())
    model = lb.LipSyncModel()
    model.load_state_dict(lb.make_synthetic_state_dict(0), strict=True)
    model.to("cuda:0").eval()
    model.compute_precision = "bf16"
    video, audio = lb.synthetic_windows(1, B)
    v = video.cuda()
    kmax = max(ks)
    _, aud = lb.synthetic_windows(2, B * kmax, t=1)
    aud = aud.view(B, kmax, *aud.shape[1:]).cuda()
    a0 = aud[:, 0].contiguous()
    plain = lambda: model(v, a0)  # noqa: E731
    with torch.no_grad():
        for _ in range(3):
            plain()
        torch.cuda.synchronize()
        res["plain_b64_ms"] = median([time_block(plain, a.window_s) for _ in range(a.reps)])
        sweeps = {}
        for K in ks:
            ak = aud[:, :K].contiguous()
            slices = [ak[:, k].contiguous() for k in range(K)]
            shared = lambda: model.forward_audio_variants(v, ak)  # noqa: E731
            naive = lambda: [model(v, s) for s in slices]  # noqa: E731
            for _ in range(2):
                shared()
                naive()
            torch.cuda.synchronize()
            out_s = shared()
            out_n = torch.stack(naive(), dim=1)
            bitwise = bool(torch.equal(out_s, out_n))
            ts, tn = [], []
            for _ in range(a.reps):
                ts.append(time_block(shared, a.window_s))
                tn.append(time_block(naive, a.window_s))
            sweeps[str(K)] = {"shared_ms": round(median(ts), 4), "naive_ms": round(median(tn), 4), "bitwise_equal": bitwise,
                              "shared_over_plain": round(median(ts) / res["plain_b64_ms"], 3),
                              "naive_over_shared": round(median(tn) / median(ts), 3),
                              "shared_ms_all": [round(x, 4) for x in ts], "naive_ms_all": [round(x, 4) for x in tn]}
    res["plain_b64_ms"] = round(res["plain_b64_ms"], 4)
    res["batch"] = B
    res["sweeps"] = sweeps
    res["timing"] = f"CUDA events, blocks of >= {a.window_s} s after warm-up, shared / naive alternating, median of {a.reps}"
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    assert all(s["bitwise_equal"] for s in sweeps.values()), "shared and naive logits differ"


if __name__ == "__main__":
    main()
