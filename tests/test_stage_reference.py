"""Every tensor-core encoder stage against a float64 reference computed from the device's own bf16 operands.

Each conv stage of the bf16 path computes y = bf16(relu(sum x*w + bias [+ residual])) with x the device's bf16 input buffer and
w = bf16(W*scale) packed with the fp32 arithmetic of pack_conv / Packer::pack_group (lsd_api.cu, bf16_path.cu).  The reference
reads the stage input back with `planar_stage`, rebuilds w bit for bit on the CPU and convolves in float64, so the kernel's only
freedom is its fp32 summation order and the final rounding:

    |dev - ref| <= REL * |ref| + C_ACC * 2^-24 * K * S,     S = sum |x|*|w| + |bias| (+ |residual|),  K = number of terms.

REL is the output rounding: 2^-8 for a bf16 stage, 2^-16 for the split-bf16 (hi, lo) audio stages, whose kernel keeps
x_hi*W_hi + x_lo*W_hi + x_hi*W_lo and drops x_lo*W_lo (Packer::add_split).  A wrong tap at a map border, a row at an M-tile
boundary or stale padding changes single elements by far more than that bound (the mutation tests below pin that), which a bound
relative to the stage maximum would not see.

The reference is evaluated on a subset of output frames: the first and last frame of every window, every frame whose folded row
(n*(T+1) + t + 1) lies within 2 rows of a multiple of 128 (the M-tiles of the folded route) and a few random ones."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# fp32 accumulation allowance: K * 2^-23 * S bounds a K-term sum in any order whose additions lose at most one fp32 ulp
# (truncating accumulation included); a single dropped tap still exceeds the bound ~25x (test_mutations_fail_the_comparator)
C_ACC = 2.0
REL_BF16, REL_SPLIT = 2.0 ** -8, 2.0 ** -16


# ---------------------------------------------------------------- geometry
def osz(i, k, s, p):
    return (i + 2 * p - k) // s + 1


def shapes(H, W, F_=80, Ta=128):
    s = {"Hs": osz(H, 7, 2, 3), "Ws": osz(W, 7, 2, 3)}
    s["H1"], s["W1"] = osz(s["Hs"], 3, 2, 1), osz(s["Ws"], 3, 2, 1)
    for i in (2, 3, 4):
        s[f"H{i}"], s[f"W{i}"] = osz(s[f"H{i-1}"], 3, 2, 1), osz(s[f"W{i-1}"], 3, 2, 1)
    s["Fs"], s["As"] = osz(F_, 7, 2, 3), osz(Ta, 7, 2, 3)
    s["F1"], s["A1"] = osz(s["Fs"], 3, 2, 1), osz(s["As"], 3, 2, 1)
    s["F2"], s["A2"] = osz(s["F1"], 3, 2, 1), osz(s["A1"], 3, 2, 1)
    s["F3"], s["A3"] = osz(s["F2"], 3, 2, 1), s["A2"]
    s["F4"], s["A4"] = osz(s["F3"], 3, 2, 1), s["A3"]
    return s


def predict_route(H, W):
    """fold_route in bf16_path.cu: a residual stage runs folded when its output map has at most 36 positions."""
    s = shapes(H, W)
    fold3, fold4 = s["H3"] * s["W3"] <= 36, s["H4"] * s["W4"] <= 36
    return "fold" if fold3 else ("mixed" if fold4 else "padded")


# (id, B, T, H, W, F, Ta, route, stages checked (None: all))
GEOMS = [
    ("fold_canonical", 5, 32, 96, 96, 80, 128, "fold", None),
    ("mixed_128", 3, 8, 128, 128, 80, 64, "mixed", None),
    ("fold_T1_64", 4, 1, 64, 64, 80, 128, "fold", None),
    ("mixed_112", 2, 8, 112, 112, 80, 127, "mixed", None),
    ("fold_odd_72", 3, 8, 72, 72, 40, 64, "fold", None),
    ("fold_T2_64", 4, 2, 64, 64, 80, 128, "fold", None),
    ("fold_100x36", 3, 8, 100, 36, 80, 72, "fold", None),
    ("padded_224", 1, 4, 224, 224, 80, 128, "padded", None),
    ("fold_many_ctas", 9, 32, 96, 96, 80, 128, "fold", ("l3a", "y3", "l4a", "y4")),
]
PADDED_96 = ("padded_96_fold_off", 2, 8, 96, 96, 80, 128, "padded", None)   # LSD_FOLD=0 (subprocess)

LAYER = "visual_encoder.layer{}"
ART = "artifact_detector.temporal_detector.temporal_conv"
# out, in, (weight, bias, bn), stride, residual, (downsample in, weight, bn, stride)
VIS_STAGES = [("l1a", "x1", (LAYER.format(1) + ".conv1.0.weight", None, LAYER.format(1) + ".conv1.1"), 1, None, None),
              ("y1", "l1a", (LAYER.format(1) + ".conv2.0.weight", None, LAYER.format(1) + ".conv2.1"), 1, "x1", None)]
for _i, _prev in ((2, "y1"), (3, "y2"), (4, "y3")):
    _p = LAYER.format(_i)
    VIS_STAGES += [(f"l{_i}a", _prev, (_p + ".conv1.0.weight", None, _p + ".conv1.1"), 2, None, None),
                   (f"y{_i}", f"l{_i}a", (_p + ".conv2.0.weight", None, _p + ".conv2.1"), 1, None,
                    (_prev, _p + ".downsample.0.weight", _p + ".downsample.1", (2, 2)))]
VIS_STAGES += [("art_a", "y4", (ART + ".0.weight", ART + ".0.bias", ART + ".1"), 1, None, None),
               ("art_b", "art_a", (ART + ".3.weight", ART + ".3.bias", ART + ".4"), 1, None, None),
               ("artd_a", "delta", (ART + ".0.weight", ART + ".0.bias", ART + ".1"), 1, None, None),
               ("artd_b", "artd_a", (ART + ".3.weight", ART + ".3.bias", ART + ".4"), 1, None, None)]
AUD = "audio_encoder.layer{}"
AUD_STAGES = []
for _i, (_prev, _st) in enumerate([("a1", (1, 1)), ("ya1", (2, 2)), ("ya2", (2, 1)), ("ya3", (2, 1))], start=1):
    _p = AUD.format(_i)
    AUD_STAGES += [(f"a{_i}a", _prev, (_p + ".conv1.0.weight", None, _p + ".conv1.1"), _st, None, None),
                   (f"ya{_i}", f"a{_i}a", (_p + ".conv2.0.weight", None, _p + ".conv2.1"), (1, 1), _prev if _i == 1 else None,
                    None if _i == 1 else (_prev, _p + ".downsample.0.weight", _p + ".downsample.1", _st))]


def stage_extents(B, T, H, W, F_, Ta):
    """True (N, T, H, W, C) of every readable stage after a forward of this geometry."""
    s = shapes(H, W, F_, Ta)
    Td = T - 1 if T > 1 else 1
    e = {"s_out": (B, T, s["Hs"], s["Ws"], 64), "x1": (B, T, s["H1"], s["W1"], 64)}
    for i, c in zip((1, 2, 3, 4), (64, 128, 256, 256)):
        e[f"l{i}a"] = e[f"y{i}"] = (B, T, s[f"H{i}"], s[f"W{i}"], c)
    e["art_a"], e["art_b"] = (B, T, s["H4"], s["W4"], 128), (B, T, s["H4"], s["W4"], 64)
    e["delta"] = (B, Td, s["H4"], s["W4"], 256)
    e["artd_a"], e["artd_b"] = (B, Td, s["H4"], s["W4"], 128), (B, Td, s["H4"], s["W4"], 64)
    e["sa_out"], e["a1"] = (B, 1, s["Fs"], s["As"], 64), (B, 1, s["F1"], s["A1"], 64)
    for i, c in zip((1, 2, 3, 4), (64, 128, 256, 256)):
        e[f"a{i}a"] = e[f"ya{i}"] = (B, 1, s[f"F{i}"], s[f"A{i}"], c)
    return e


AUDIO_NAMES = ("sa_out", "a1", "a1a", "ya1", "a2a", "ya2", "a3a", "ya3", "a4a", "ya4")


def read_stages(model, geom, names=None):
    """fp32 numpy copies of the stages (audio stages: the high part and the (hi + lo) sum)."""
    _, B, T, H, W, F_, Ta, _, _ = geom
    out = {}
    for name, shape in stage_extents(B, T, H, W, F_, Ta).items():
        if names is not None and name not in names:
            continue
        out[name] = model.planar_stage(name, shape).cpu().numpy()
        if name in AUDIO_NAMES:
            out[name + "+lo"] = model.planar_stage(name, shape, lo=name + "_lo").cpu().numpy()
    return out


def needed(only):
    """Stages to read when only `only` is checked: those and their inputs."""
    if only is None:
        return None
    specs = [sp for sp in VIS_STAGES if sp[0] in only]
    return set(only) | {sp[1] for sp in specs} | {sp[4] for sp in specs if sp[4]} | {sp[5][0] for sp in specs if sp[5]}


def pick_frames(B, T, seed=0, n_random=3):
    fr = {(n, t) for n in range(B) for t in (0, T - 1)}
    for n in range(B):
        for t in range(T):
            row = n * (T + 1) + t + 1
            if min(row % 128, 128 - row % 128) <= 2:
                fr.add((n, t))
    rng = np.random.default_rng(seed)
    for _ in range(n_random):
        fr.add((int(rng.integers(B)), int(rng.integers(T))))
    return sorted(fr)


# ---------------------------------------------------------------- the packer's arithmetic
def f2bf_bits(v):
    """f2bf (bf16_path.cu) restated: round-to-nearest-even on the fp32 bit pattern, Inf / NaN passed through."""
    u = np.ascontiguousarray(v, dtype=np.float32).view(np.uint32)
    r = ((u + np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))) >> np.uint32(16)).astype(np.uint16)
    return np.where((u & np.uint32(0x7F800000)) == np.uint32(0x7F800000), (u >> np.uint32(16)).astype(np.uint16), r)


def bf16(a):
    """float32 array -> its bf16 rounding (RN), as float64 torch."""
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(torch.bfloat16).double()


def folded(sd, wkey, bkey, bn, exact=False):
    """pack_conv: scale = gamma / sqrtf(var + 1e-5f), shift = beta - mean*scale (+ bias*scale), v = W*scale, in fp32
    (float64 when exact).  -> (v (Cout, Cin, k...), shift (Cout,)) as numpy."""
    dt = np.float64 if exact else np.float32
    W = sd[wkey].numpy().astype(dt)
    g, be, mu, var = (sd[bn + s].numpy().astype(dt) for s in (".weight", ".bias", ".running_mean", ".running_var"))
    sc = g / np.sqrt(var + dt(1e-5))
    shift = be - mu * sc
    if bkey is not None:
        shift = shift + sd[bkey].numpy().astype(dt) * sc
    return W * sc.reshape((-1,) + (1,) * (W.ndim - 1)), shift


_WCACHE = {}


def weights(sd, wkey, bkey, bn, mode):
    """Weight terms of a conv: mode "bf16" -> [w_hi]; "split" -> [w_hi, w_lo]; "exact" -> [float64 W*scale]; + shift."""
    key = (id(sd), wkey, mode)
    if key not in _WCACHE:
        v, shift = folded(sd, wkey, bkey, bn, exact=mode == "exact")
        if mode == "exact":
            ws = [torch.from_numpy(v)]
        else:
            hi = bf16(v)
            ws = [hi] + ([bf16(v - hi.float().numpy())] if mode == "split" else [])
        ws = [w if w.dim() == 5 else w.unsqueeze(2) for w in ws]   # 2-D audio convs as kt = 1
        _WCACHE[key] = (ws, torch.from_numpy(np.asarray(shift, dtype=np.float64)))
    return _WCACHE[key]


# ---------------------------------------------------------------- float64 reference on selected frames
def _slabs(x, frames, kt):
    """x (N, T, H, W, C) -> (frames, C, kt, H, W): the kt-frame input slab of each output frame, zero outside the window."""
    T = x.shape[1]
    out = torch.zeros((len(frames), kt) + tuple(x.shape[2:]), dtype=torch.float64)
    for i, (n, t) in enumerate(frames):
        for a in range(kt):
            if 0 <= t + a - kt // 2 < T:
                out[i, a] = x[n, t + a - kt // 2]
    return out.permute(0, 4, 1, 2, 3)


def _conv(terms, frames, stride, pad):
    """sum over (x, w) terms of conv(x, w) and of conv(|x|, |w|) at the selected frames -> two (frames, Ho, Wo, Cout)."""
    acc = S = 0
    for x, w in terms:
        sl = _slabs(x, frames, w.shape[2])
        kw = dict(stride=(1,) + tuple(stride), padding=(0,) + tuple(pad))
        acc = acc + F.conv3d(sl, w, **kw)
        S = S + F.conv3d(sl.abs(), w.abs(), **kw)
    return acc[:, :, 0].permute(0, 2, 3, 1), S[:, :, 0].permute(0, 2, 3, 1)


def _terms(xs, ws):
    """(x parts, w parts) -> products the kernel sums: x*w, or x_hi*W_hi + x_lo*W_hi + x_hi*W_lo for split operands."""
    if len(xs) == 1:
        return [(xs[0], ws[0])]
    return [(xs[0], ws[0]), (xs[1], ws[0]), (xs[0], ws[1])]


def stage_reference(sd, spec, get, frames, mode):
    """-> (ref, S, K) of stage `spec` at `frames`; get(name) -> the (N, T, H, W, C) parts of a stage buffer (one, or hi and lo)."""
    out, src, (wkey, bkey, bn), stride, res, ds = spec
    stride = (stride, stride) if isinstance(stride, int) else stride
    ws, shift = weights(sd, wkey, bkey, bn, mode)
    xs = get(src)
    terms = _terms(xs, ws)
    pad = (ws[0].shape[3] // 2, ws[0].shape[4] // 2)
    acc, S = _conv(terms, frames, stride, pad)
    K = len(terms) * ws[0][0].numel()
    acc, S = acc + shift, S + shift.abs()
    if ds is not None:
        dws, dshift = weights(sd, ds[1], None, ds[2], mode)
        dterms = _terms(get(ds[0]), dws)
        a2, s2 = _conv(dterms, frames, ds[3], (0, 0))
        acc, S, K = acc + a2 + dshift, S + s2 + dshift.abs(), K + len(dterms) * dws[0][0].numel()
    if res is not None:
        r = torch.stack([sum(p[n, t].double() for p in get(res)) for n, t in frames])
        acc, S, K = acc + r, S + r.abs(), K + 1
    return torch.relu(acc), S, K


def ratio(dev, ref, S, K, rel):
    """Largest |dev - ref| / (rel*|ref| + C_ACC*2^-24*K*S); an element with a zero bound must match exactly."""
    dev, ref, S = (np.asarray(a, dtype=np.float64) for a in (dev, ref, S))
    err = np.abs(dev - ref)
    bound = rel * np.abs(ref) + C_ACC * 2.0 ** -24 * K * S
    r = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))
    return float(r.max()) if r.size else 0.0


# ---------------------------------------------------------------- checks of one forward
def visual_stem_input(video):
    """video (B, 3, T, H, W) fp32 -> the stem's bf16 operand (RN, video_rows) as (B, T, H, W, 3) float64."""
    return bf16(video.permute(0, 2, 3, 4, 1).contiguous().numpy())


def check_forward(sd, geom, stages, video, audio, report):
    """All stage checks of one forward; report[stage] = worst error / bound, or for the bit-exact stages (x1, delta, a1) the
    number of elements that differ."""
    gid, B, T, H, W, F_, Ta, route, only = geom
    frames = pick_frames(B, T, seed=B * 1000 + T)

    def want(name):
        return only is None or name in only

    if want("s_out"):
        stem = ("s_out", "video", ("visual_encoder.stem.0.weight", None, "visual_encoder.stem.1"), 2, None, None)
        ref, S, K = stage_reference(sd, stem, lambda n: [visual_stem_input(video)], frames, "bf16")
        dev = np.stack([stages["s_out"][n, t] for n, t in frames])
        report["s_out"] = ratio(dev, ref.numpy(), S.numpy(), K, REL_BF16)
    if want("x1"):
        so = torch.from_numpy(stages["s_out"]).permute(0, 1, 4, 2, 3).reshape(B * T, 64, *stages["s_out"].shape[2:4])
        x1 = F.max_pool2d(so, 3, 2, 1).reshape(B, T, 64, *stages["x1"].shape[2:4]).permute(0, 1, 3, 4, 2).numpy()
        report["x1"] = float(np.count_nonzero(x1 != stages["x1"]))
    if want("delta"):
        y4 = stages["y4"]
        d = (y4[:, 1:] - y4[:, :-1]) if T > 1 else np.zeros_like(y4)
        d = bf16(d).float().numpy()
        report["delta"] = float(np.count_nonzero(d != stages["delta"]))
    for spec in VIS_STAGES:
        name = spec[0]
        if not want(name):
            continue
        fr = frames if not name.startswith("artd") else pick_frames(B, max(T - 1, 1), seed=B)
        ref, S, K = stage_reference(sd, spec, lambda n: [torch.from_numpy(stages[n])], fr, "bf16")
        dev = np.stack([stages[name][n, t] for n, t in fr])
        report[name] = ratio(dev, ref.numpy(), S.numpy(), K, REL_BF16)
    if only is not None:
        return
    # audio encoder: (hi, lo) pairs, whole maps
    afr = [(n, 0) for n in range(B)]
    parts = {k: [torch.from_numpy(stages[k]).double(), torch.from_numpy(stages[k + "+lo"] - stages[k]).double()] for k in AUDIO_NAMES}
    a = audio.permute(0, 2, 3, 1).unsqueeze(1).contiguous().numpy()   # (B, 1, F, Ta, 1)
    ahi = bf16(a)
    alo = bf16(a - ahi.float().numpy())
    stem = ("sa_out", "audio", ("audio_encoder.stem.0.weight", None, "audio_encoder.stem.1"), (2, 2), None, None)
    ref, S, K = stage_reference(sd, stem, lambda n: [ahi, alo], afr, "split")
    report["sa_out"] = ratio(stages["sa_out+lo"][:, 0], ref.numpy(), S.numpy(), K, REL_SPLIT)
    so = torch.from_numpy(stages["sa_out+lo"][:, 0]).permute(0, 3, 1, 2)
    a1 = F.max_pool2d(so, 3, 2, 1).permute(0, 2, 3, 1).numpy()
    report["a1"] = float(np.count_nonzero(a1 != stages["a1+lo"][:, 0]))
    for spec in AUD_STAGES:
        ref, S, K = stage_reference(sd, spec, lambda n: parts[n], afr, "split")
        report[spec[0]] = ratio(stages[spec[0] + "+lo"][:, 0], ref.numpy(), S.numpy(), K, REL_SPLIT)


def _inputs(geom, seed):
    import lipsync_b200 as lb
    _, B, T, H, W, F_, Ta, _, _ = geom
    return lb.synthetic_windows(seed, B, T, H, W, F_, Ta)


def _assert_report(gid, report):
    print(f"{gid}: worst error / bound per stage:", json.dumps({k: round(v, 4) for k, v in report.items()}))
    bad = {k: v for k, v in report.items() if not v < 1.0}
    assert not bad, (gid, bad)


# ---------------------------------------------------------------- CPU: the reference itself
@pytest.fixture(scope="module")
def sd0():
    import lipsync_b200 as lb
    return lb.make_synthetic_state_dict(0)


def test_route_prediction():
    for gid, B, T, H, W, *_rest in GEOMS + [PADDED_96]:
        route = _rest[-2]
        s = shapes(H, W)
        expect = "fold" if s["H3"] * s["W3"] <= 36 else ("mixed" if s["H4"] * s["W4"] <= 36 else "padded")
        if gid == PADDED_96[0]:
            assert predict_route(H, W) == "fold"       # padded only because LSD_FOLD=0
            continue
        assert predict_route(H, W) == expect == route, gid
    assert (shapes(72, 72)["H2"], shapes(72, 72)["H3"], shapes(72, 72)["H4"]) == (9, 5, 3)
    s = shapes(100, 36)
    assert [(s[f"H{i}"], s[f"W{i}"]) for i in (2, 3, 4)] == [(13, 5), (7, 3), (4, 2)]
    assert (shapes(112, 112)["H3"], shapes(112, 112)["H4"]) == (7, 4)


def test_frame_pick_covers_tile_boundaries():
    fr = pick_frames(5, 32)
    rows = {n * 33 + t + 1 for n, t in fr}
    assert {126, 127, 128, 129, 130} <= rows            # boundary inside window 3 (rows 100 .. 131)
    assert all((n, 0) in fr and (n, 31) in fr for n in range(5))
    rows9 = {n * 33 + t + 1 for n, t in pick_frames(9, 32)}
    assert {127, 128, 129, 255, 256, 257} <= rows9


def test_reproduced_weights_match_the_packer(sd0):
    """bf16(W*scale) via numpy fp32 + torch RN equals a line-for-line restatement of pack_conv (arena [tap][ci][co], fp32 scale)
    and Packer::pack_group (f2bf of W*scale; the low part f2bf(v - hi))."""
    for wkey, bn in [("visual_encoder.stem.0.weight", "visual_encoder.stem.1"), (LAYER.format(3) + ".conv2.0.weight", LAYER.format(3) + ".conv2.1"),
                     (LAYER.format(2) + ".downsample.0.weight", LAYER.format(2) + ".downsample.1"), (AUD.format(2) + ".conv1.0.weight", AUD.format(2) + ".conv1.1")]:
        w = sd0[wkey].numpy().astype(np.float32)
        Cout, Cin = w.shape[:2]
        taps = int(np.prod(w.shape[2:]))
        arena = np.empty((taps, Cin, Cout), np.float32)
        for co in range(Cout):
            for ci in range(Cin):
                arena[:, ci, co] = w.reshape(Cout, Cin, taps)[co, ci]
        g, be, mu, var = (sd0[bn + s].numpy().astype(np.float32) for s in (".weight", ".bias", ".running_mean", ".running_var"))
        sc = np.array([g[i] / np.float32(np.sqrt(np.float32(var[i] + np.float32(1e-5)))) for i in range(Cout)], np.float32)
        v = arena * sc[None, None, :]
        hi_bits = f2bf_bits(v)
        hf = (hi_bits.astype(np.uint32) << np.uint32(16)).view(np.float32)
        lo_bits = f2bf_bits(v - hf)
        (whi, wlo), _ = weights(sd0, wkey, None, bn, "split")
        ref_hi = whi.float().reshape(Cout, Cin, taps).permute(2, 1, 0).contiguous().to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
        ref_lo = wlo.float().reshape(Cout, Cin, taps).permute(2, 1, 0).contiguous().to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
        assert np.array_equal(hi_bits, ref_hi), wkey
        assert np.array_equal(lo_bits, ref_lo), wkey
    # f2bf itself: ties to even, Inf / NaN kept
    x = np.array([1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -2.5, np.inf, 3.0e38], np.float32)
    assert np.array_equal(f2bf_bits(x), torch.from_numpy(x).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16))


def _sd64(sd):
    return {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}


@pytest.mark.parametrize("hw", [(96, 96), (128, 128), (224, 224)])
def test_reference_equals_oracle_visual(sd0, hw):
    """With rounding switched off (float64 W*scale, float64 inputs) the stage reference reproduces the oracle's visual encoder
    stage by stage, fed the oracle's own inputs: pins BN folding, strides, padding, downsample and residual wiring."""
    from oracle import lipsync_oracle as orc
    H, W = hw
    sd64 = _sd64(sd0)
    g = torch.Generator().manual_seed(5)
    B, T = 1, 3
    video = torch.rand((B, 3, T, H, W), generator=g, dtype=torch.float64)
    inter = {}
    orc.visual_encoder(sd64, video, inter)
    cl = lambda x: x.permute(0, 2, 3, 4, 1).contiguous()
    st = {"video": cl(video), "s_out": cl(inter["v_stem_conv"]), "x1": cl(inter["v_stem"])}
    for i, stride in zip((1, 2, 3, 4), (1, 2, 2, 2)):
        p = LAYER.format(i)
        xin = st["x1"] if i == 1 else st[f"y{i-1}"]
        mid = F.relu(orc._bn(sd64, p + ".conv1.1", F.conv3d(cl_inv(xin), sd64[p + ".conv1.0.weight"], stride=(1, stride, stride), padding=1)))
        st[f"l{i}a"], st[f"y{i}"] = cl(mid), cl(inter[f"v_layer{i}"])
    fmap = inter["v_layer4"]
    for pre, x in (("art", fmap), ("artd", fmap[:, :, 1:] - fmap[:, :, :-1])):
        a = F.relu(orc._bn(sd64, ART + ".1", F.conv3d(x, sd64[ART + ".0.weight"], sd64[ART + ".0.bias"], padding=1)))
        b = F.relu(orc._bn(sd64, ART + ".4", F.conv3d(a, sd64[ART + ".3.weight"], sd64[ART + ".3.bias"], padding=1)))
        st[pre + "_a"], st[pre + "_b"] = cl(a), cl(b)
        st["delta" if pre == "artd" else "_"] = cl(x)
    stem = ("s_out", "video", ("visual_encoder.stem.0.weight", None, "visual_encoder.stem.1"), 2, None, None)
    for spec in [stem] + VIS_STAGES:
        Tn = st[spec[1]].shape[1]
        frames = [(0, t) for t in range(Tn)]
        ref, _, _ = stage_reference(sd0, spec, lambda n: [st[n]], frames, "exact")
        want = torch.stack([st[spec[0]][0, t] for _, t in frames])
        rel = float((ref - want).abs().max()) / float(want.abs().max())
        assert rel <= 1e-6, (spec[0], rel)


def cl_inv(x):
    return x.permute(0, 4, 1, 2, 3).contiguous()


@pytest.mark.parametrize("fta", [(80, 128), (40, 64), (80, 127)])
def test_reference_equals_oracle_audio(sd0, fta):
    from oracle import lipsync_oracle as orc
    F_, Ta = fta
    sd64 = _sd64(sd0)
    g = torch.Generator().manual_seed(6)
    audio = -80.0 * torch.rand((2, 1, F_, Ta), generator=g, dtype=torch.float64)
    inter = {}
    orc.audio_encoder(sd64, audio, inter)
    cl = lambda x: x.permute(0, 2, 3, 1).unsqueeze(1).contiguous()     # (B, C, F, T) -> (B, 1, F, T, C)
    st = {"audio": cl(audio), "a1": cl(inter["a_stem"])}
    for i, stride in zip((1, 2, 3, 4), ((1, 1), (2, 2), (2, 1), (2, 1))):
        p = AUD.format(i)
        xin = inter["a_stem"] if i == 1 else inter[f"a_layer{i-1}"]
        st[f"a{i}a"] = cl(F.relu(orc._bn(sd64, p + ".conv1.1", F.conv2d(xin, sd64[p + ".conv1.0.weight"], stride=stride, padding=1))))
        st[f"ya{i}"] = cl(inter[f"a_layer{i}"])
    for spec in AUD_STAGES:
        frames = [(n, 0) for n in range(2)]
        ref, _, _ = stage_reference(sd0, spec, lambda n: [st[n]], frames, "exact")
        want = st[spec[0]][:, 0]
        rel = float((ref - want).abs().max()) / float(want.abs().max())
        assert rel <= 1e-6, (spec[0], rel)


def test_mutations_fail_the_comparator(sd0):
    """A reference with one in-bounds tap dropped at a border output position, or the output of the neighbouring frame, must
    fail the bound at every map size of the geometry table: C_ACC is below the value at which a single dropped tap would pass."""
    g = torch.Generator().manual_seed(11)
    sizes = set()
    for gid, B, T, H, W, *_ in GEOMS:
        s = shapes(H, W)
        for i in (1, 2, 3, 4):
            sizes.add((i, s[f"H{i}"], s[f"W{i}"]))
    least_drop = np.inf
    for layer, Ho, Wo in sorted(sizes):
        conv2 = next(sp for sp in VIS_STAGES if sp[0] == f"y{layer}")
        ws, shift = weights(sd0, conv2[2][0], None, conv2[2][2], "bf16")
        w = ws[0]
        Cout, Cin = w.shape[:2]
        x = bf16(torch.relu(torch.randn((1, 3, Ho, Wo, Cin), generator=g)).numpy())
        frames = [(0, 1)]
        spec = (f"y{layer}", "in", conv2[2], 1, None, None)
        ref, S, K = stage_reference(sd0, spec, lambda n: [x], frames, "bf16")
        # the "device": fp32 accumulation, bf16 output
        sl = _slabs(x, frames, 3).float()
        dev = bf16(torch.relu(F.conv3d(sl, w.float(), padding=(0, 1, 1))[:, :, 0].permute(0, 2, 3, 1) + shift.float()).numpy()).numpy()
        assert ratio(dev, ref.numpy(), S.numpy(), K, REL_BF16) < 1.0, (layer, Ho, Wo)
        # drop the in-bounds tap (kt=1, kh=2, kw=2) of the bottom-right corner output position
        acc, _ = _conv([(x, w)], frames, (1, 1), (1, 1))
        pre = acc + shift
        h, ww = Ho - 1, Wo - 1
        tap = (x[0, 1, h - 1 if Ho > 1 else h, ww - 1 if Wo > 1 else ww] @ w[:, :, 1, 0 if Ho > 1 else 1, 0 if Wo > 1 else 1].t())
        mut = pre.clone()
        mut[0, h, ww] -= tap
        r_drop = ratio(dev, torch.relu(mut).numpy(), S.numpy(), K, REL_BF16)
        least_drop = min(least_drop, r_drop)
        assert r_drop > 1.0, ("dropped tap passes", layer, Ho, Wo, r_drop)
        # the neighbouring frame's output in place of this one
        ref2, S2, _ = stage_reference(sd0, spec, lambda n: [x], [(0, 2)], "bf16")
        assert ratio(dev, ref2.numpy(), S2.numpy(), K, REL_BF16) > 1.0, ("frame shift passes", layer, Ho, Wo)
    print("smallest error / bound of a dropped tap:", round(least_drop, 2))


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def gpu_model(sd0):
    import __graft_entry__ as ge
    ge.build()
    import lipsync_b200 as lb
    m = lb.LipSyncModel()
    m.load_state_dict(sd0, strict=True)
    m = m.to("cuda:0").eval()
    m.compute_precision = "bf16"
    return m


@pytest.mark.gpu
def test_planar_stage_read_rejects_wrong_extents(gpu_model):
    """lsd_planar_stage_read accepts only the true map extent of a buffer (any layout: plain, parity-split, folded) and a low
    part of the same layout; everything else returns its status on the host, before anything is launched."""
    import lipsync_b200 as lb
    from lipsync_b200 import _cabi as cabi
    m = gpu_model
    L = cabi.lib()
    h = m._ensure_handle(m._device())

    def read(name, shape, lo=None):
        out = torch.empty(shape, dtype=torch.float32, device="cuda")
        return L.lsd_planar_stage_read(h.ptr, name.encode(), lo.encode() if lo else None, m._lsd_ws.data_ptr(), out.data_ptr(),
                                       out.numel(), int(shape[2]), int(shape[3]), None)

    v, a = lb.synthetic_windows(3, 2, 8, 100, 36)
    m(v.cuda(), a.cuda())
    torch.cuda.synchronize()
    n0 = m.launch_count()
    assert read("x1", (2, 8, 24, 9, 64)) == cabi.LSD_ERR_SHAPE          # wrong extent (25 x 9) of a plain buffer
    assert read("y1", (2, 8, 9, 25, 64)) == cabi.LSD_ERR_SHAPE          # swapped H / W
    assert read("l1a", (2, 8, 9, 25, 64)) == cabi.LSD_ERR_SHAPE
    assert read("y1", (2, 8, 26, 9, 64)) == cabi.LSD_ERR_SHAPE          # parity buffer read with Hf + 1
    assert read("ya2", (2, 1, 11, 16, 128), lo="ya2_lo") == cabi.LSD_ERR_SHAPE
    assert read("ya4", (2, 1, 3, 16, 256), lo="y4") == cabi.LSD_ERR_SHAPE          # low part of another layout
    assert read("xs", (2, 8, 50, 18, 8)) == cabi.LSD_ERR_ARG            # pixel rows are not a channel map
    assert read("nope", (2, 8, 1, 1, 8)) == cabi.LSD_ERR_ARG
    v, a = lb.synthetic_windows(3, 2, 32, 64, 64)
    m(v.cuda(), a.cuda())
    torch.cuda.synchronize()
    n1 = m.launch_count()
    assert read("y3", (2, 32, 6, 6, 256)) == cabi.LSD_ERR_SHAPE         # folded 4 x 4 buffer read with the 96x96 extent
    assert read("l4a", (2, 32, 3, 3, 256)) == cabi.LSD_ERR_SHAPE
    assert read("y3", (2, 32, 4, 4, 128)) == cabi.LSD_ERR_SHAPE         # right extent, wrong element count
    assert m.launch_count() == n1
    assert read("y3", (2, 32, 4, 4, 256)) == cabi.LSD_OK                # the true extent reads (one launch)
    assert m.launch_count() == n1 + 1
    assert n1 > n0


@pytest.mark.gpu
def test_stages_against_same_operand_reference(gpu_model, sd0):
    """Fold -> mixed -> fold -> padded -> fold geometries through one model handle: every stage of every geometry within its
    same-operand bound, the max-pool and the temporal delta bit for bit."""
    m = gpu_model
    for geom in GEOMS:
        assert predict_route(geom[3], geom[4]) == geom[7]
        video, audio = _inputs(geom, 7)
        m(video.cuda(), audio.cuda())
        stages = read_stages(m, geom, needed(geom[8]))
        report = {}
        check_forward(sd0, geom, stages, video, audio, report)
        _assert_report(geom[0], report)


SUB = """
import sys; sys.path.insert(0, %r)
import numpy as np, torch, lipsync_b200 as lb
from tests.test_stage_reference import read_stages, _inputs, GEOMS, PADDED_96
m = lb.LipSyncModel(); m.load_state_dict(lb.make_synthetic_state_dict(0)); m.to('cuda:0').eval(); m.compute_precision = 'bf16'
for geom in [PADDED_96, [g for g in GEOMS if g[0] == 'mixed_128'][0]]:
    v, a = _inputs(geom, 7)
    m(v.cuda(), a.cuda())
    np.savez(%r + geom[0] + '.npz', **read_stages(m, geom))
"""


def _subprocess_stages(env, prefix):
    r = subprocess.run([sys.executable, "-c", SUB % (ROOT, prefix)], env={**os.environ, **env}, capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    return {g: dict(np.load(prefix + g + ".npz")) for g in (PADDED_96[0], "mixed_128")}


@pytest.mark.gpu
def test_padded_route_and_flat_stem_against_reference(gpu_model, sd0, tmp_path):
    """LSD_FOLD=0 (padded layer3 / layer4 at 96x96 and 128x128) and LSD_STEM_RING=0 (flat shift-GEMM stem): the knobs are read
    once per process, so each runs in a fresh interpreter.  At 128x128 layer3 runs padded on both routes, so y3 is bit for bit
    the mixed route's; y4 (folded vs padded layer4) agrees within the stage bound."""
    mixed = [g for g in GEOMS if g[0] == "mixed_128"][0]
    padded = _subprocess_stages({"LSD_FOLD": "0"}, str(tmp_path / "fold0_"))
    flat = _subprocess_stages({"LSD_STEM_RING": "0"}, str(tmp_path / "flat_"))
    for tag, runs in (("fold_off", padded), ("flat_stem", flat)):
        for geom in (PADDED_96, mixed):
            report = {}
            video, audio = _inputs(geom, 7)
            check_forward(sd0, geom, runs[geom[0]], video, audio, report)
            _assert_report(f"{geom[0]}[{tag}]", report)
    # same input, mixed route in this process
    video, audio = _inputs(mixed, 7)
    gpu_model(video.cuda(), audio.cuda())
    here = read_stages(gpu_model, mixed, {"y3", "l4a", "y4"})
    p = padded["mixed_128"]
    assert np.array_equal(here["y3"], p["y3"])
    B, T = mixed[1], mixed[2]
    frames = pick_frames(B, T)
    y4spec = next(sp for sp in VIS_STAGES if sp[0] == "y4")
    ref, S, K = stage_reference(sd0, y4spec, lambda n: [torch.from_numpy(here[n])], frames, "bf16")
    r = ratio(np.stack([p["y4"][n, t] for n, t in frames]), np.stack([here["y4"][n, t] for n, t in frames]), S.numpy(), K, REL_BF16)
    print("y4 mixed vs padded route: worst difference / stage bound", round(r, 4))
    assert r < 1.0
