"""Window-scoring API: the scoring/aggregation subset of the reference `Predictor`
(app/inference/predictor.py), re-hosted on the batched B200 forward.

Mirrors, with the reference's names, argument meaning and return values:
  `_infer_confidence`              predictor.py:212-244   (+ batched `_infer_confidences`)
  `_robust_confidence`             predictor.py:246-260
  `_speech_weighted_confidence`    predictor.py:262-293
  `_temporal_smoothed_confidence`  predictor.py:295-331
  `_align_audio_chunk`             predictor.py:525-552
  `_run_chunked_inference`         predictor.py:554-580   (serial B=1 loop -> batches of `batch_size` windows)
New (SURVEY.md §8e/f): `score_track` (uint8 track -> device-built windows, C `lsd_score_windows`) and
`score_windows_sharded` (contiguous block partition over ranks + one all-gather of fp32 logits).
Video decode, face tracking, VAD and the gate/verdict block of `_predict_long_video` stay reference Python.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import time
from fractions import Fraction
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _cabi
from . import aggregate as _agg
from .model import LipSyncModel

#: one log-mel column: hop 160 at 16 kHz (app/preprocessing/audio.py:80-91)
_MEL_HOP_SEC = 160.0 / 16000.0


def partition_windows(n_windows: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous block partition of [0, n_windows): rank r owns [lo, hi) with ceil(n/R) windows per rank
    (SURVEY.md §8e: contiguous so each rank reads one contiguous span of the track)."""
    per = -(-n_windows // world_size) if world_size > 0 else n_windows
    lo = min(n_windows, rank * per)
    hi = min(n_windows, lo + per)
    return lo, hi


def gather_logits(local: torch.Tensor, n_windows: int, world_size: int, rank: int) -> torch.Tensor:
    """All-gather per-rank fp32 logits (padded to ceil(n/R)) and strip the padding: the only collective on the path."""
    import torch.distributed as dist

    per = -(-n_windows // world_size)
    buf = torch.zeros(per, dtype=torch.float32, device=local.device)
    buf[: local.numel()] = local.to(torch.float32)
    if world_size == 1:
        return buf[:n_windows]
    out = torch.empty(world_size * per, dtype=torch.float32, device=local.device)
    if local.is_cuda:
        dist.all_gather_into_tensor(out, buf)  # NCCL over NVLink: <= 4 B per window
    else:
        dist.all_gather(list(out.view(world_size, per).unbind(0)), buf)  # gloo (CPU tests of the host logic)
    return out[:n_windows]


def auto_transport_gives_up_packing(steady_ms: Sequence[float], all_ms: Sequence[float], t32_s: float) -> bool:
    """The decision of `host_transport="auto"` (a pure function of the measured pack times, unit-tested on CPU): stop packing when
    packing is the slower way to feed the GPU.  `steady_ms`: whole-batch pack times in ms, oldest first, without the first batch of a
    call and without first packs into freshly pinned staging buffers; `all_ms`: every pack but the very first of the predictor;
    `t32_s`: the fp32 bytes of a batch at ~52 GB/s of PCIe gen5 x16, in seconds.
      * marginal: the fastest of the last three steady packs (once four are measured) + 0.1 ms is slower than the fp32 copy — a slow
        pack or two on a busy host must not flip the transport for good;
      * clearly slower: the last two packs of any kind both took more than 1.5 x the fp32 copy (every GPU of a box fed at once: the
        host DRAM is the limit and the pack moves more of it than the copy it saves — 12 ms against 4.4 ms with eight GPUs) — decided
        within a three-batch warm-up call instead of five batches into the next one."""
    if len(steady_ms) >= 4 and min(steady_ms[-3:]) * 1e-3 + 0.1e-3 > t32_s:
        return True
    return len(all_ms) >= 2 and min(all_ms[-2:]) * 1e-3 > 1.5 * t32_s


class Predictor:
    """Scoring half of the reference Predictor.  `model` is a `lipsync_b200.LipSyncModel` already on a CUDA device."""

    def __init__(
        self,
        model: LipSyncModel,
        device: Optional[torch.device] = None,
        use_half_precision: bool = False,
        confidence_smoothing: str = "median",
        trim_ratio: float = 0.1,
        calibration_method: str = "none",
        calibration_temperature: float = 1.0,
        calibration_platt_a: float = 1.0,
        calibration_platt_b: float = 0.0,
        isotonic_calibrator=None,
        chunk_size: int = 32,
        chunk_stride: int = 8,
        batch_size: int = 64,
        use_cuda_graphs: bool = True,
        graph_max_batch: int = 8,
        host_transport: str = "auto",
        host_pack_threads: Optional[int] = None,
        host_split: bool = False,
    ) -> None:
        self.model = model
        self.device = device if device is not None else (model._device() if model is not None else torch.device("cpu"))
        self.use_half_precision = bool(use_half_precision and self.device.type == "cuda")
        allowed = {"none", "median", "trimmed_mean"}
        self.confidence_smoothing = confidence_smoothing if confidence_smoothing in allowed else "median"
        self.trim_ratio = float(min(max(trim_ratio, 0.0), 0.49))
        _cal_allowed = {"none", "temperature", "platt", "isotonic"}
        self._cal_method = calibration_method if calibration_method in _cal_allowed else "none"
        self._cal_temperature = float(max(1e-3, calibration_temperature))
        self._cal_platt_a = float(calibration_platt_a)
        self._cal_platt_b = float(calibration_platt_b)
        self._isotonic_cal = isotonic_calibrator
        if self._cal_method == "isotonic" and self._isotonic_cal is None:
            self._cal_method = "none"
        self.chunk_size = int(chunk_size)
        self.chunk_stride = int(chunk_stride)
        self.batch_size = int(max(1, batch_size))
        #: small host batches (the B=1 calls of `_infer_confidence`, the 1+3 windows of `_temporal_smoothed_confidence`) replay a
        #: captured CUDA graph (H2D copies + the ~60 launches of the forward + D2H) instead of enqueueing launch by launch
        self.use_cuda_graphs = bool(use_cuda_graphs)
        self.graph_max_batch = int(graph_max_batch)
        self._graphs = {}
        self.graph_captures = 0      # how many graphs this predictor captured (a rising count under steady shapes = re-capture churn)
        #: how fp32 host windows cross PCIe in `score_batches`: "u8" packs windows whose pixels are exactly k/255 (what
        #: video.py:552-556 produces) to one byte per pixel on the host threads (`lsd_host_pack_u8_exact`: verified value by value,
        #: logits bit-identical), "fp32" copies them as they are, "auto" packs when the first batch qualifies and keeps packing
        #: unless the pack turns out slower than PCIe would move the fp32 bytes (fastest of the last three packs once four are measured, remembered across calls, see finish())
        if host_transport not in ("auto", "u8", "fp32"):
            raise ValueError(f"host_transport must be 'auto', 'u8' or 'fp32', got {host_transport!r}")
        self.host_transport = host_transport
        #: split transport of `score_batches` (opt-in): part of every batch crosses PCIe as fp32 while the host threads pack the rest
        #: (True: the share follows the measured pack rate; a float in (0, 1) fixes it; logits unchanged, `lsd_expand_u8`).  Off by
        #: default: measured slower than packing whole batches on one GPU (17.1 k against 22 k windows/s end to end, and unstable —
        #: the fp32 part and the pack threads read the same host DRAM at once).
        self.host_split = host_split if isinstance(host_split, float) else bool(host_split)
        if host_pack_threads is None:
            local_ws = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
            try:
                cpus = len(os.sched_getaffinity(0))
            except (AttributeError, OSError):
                cpus = os.cpu_count() or 1
            host_pack_threads = max(1, min(32, cpus // local_ws))
        self.host_pack_threads = int(host_pack_threads)
        self.last_transport = "fp32"
        self.last_h2d_bytes_per_batch = 0

    # ------------------------------------------------------------------ calibration (predictor.py:226-244)
    def _calibrate(self, logit_val: float) -> float:
        if self._cal_method == "temperature":
            return float(torch.sigmoid(torch.tensor(logit_val / self._cal_temperature)).item())
        if self._cal_method == "platt":
            return float(torch.sigmoid(torch.tensor(self._cal_platt_a * logit_val + self._cal_platt_b)).item())
        raw_prob = float(torch.sigmoid(torch.tensor(logit_val, dtype=torch.float32)).item())
        if self._cal_method == "isotonic" and self._isotonic_cal is not None:
            cal_prob = float(self._isotonic_cal.predict([[raw_prob]])[0])
            return float(np.clip(cal_prob, 0.0, 1.0))
        return raw_prob

    # ------------------------------------------------------------------ scoring
    def _infer_logits(self, visuals: Sequence[np.ndarray], audios: Sequence[np.ndarray]) -> List[float]:
        """Batched forward over host windows of one common shape, `batch_size` windows per launch."""
        n = len(visuals)
        if (self.use_cuda_graphs and 0 < n <= self.graph_max_batch and self.model is not None and self.device.type == "cuda"
                and self.model._precision() == _cabi.LSD_PREC_BF16):
            return self._infer_logits_graph(visuals, audios)

        def gen():
            for i0 in range(0, n, self.batch_size):
                v = torch.from_numpy(np.stack(visuals[i0:i0 + self.batch_size])).pin_memory()
                a = torch.from_numpy(np.stack(audios[i0:i0 + self.batch_size])).pin_memory()
                yield v, a

        out: List[float] = []
        for t in self.score_batches(gen()):
            out.extend(float(x) for x in t.tolist())
        return out

    # ------------------------------------------------------------------ CUDA-graph path for small host batches
    def _infer_logits_graph(self, visuals: Sequence[np.ndarray], audios: Sequence[np.ndarray]) -> List[float]:
        """`len(visuals) <= graph_max_batch` host windows of one shape -> logits, through a CUDA graph captured once per
        (batch, shapes, dtype): pinned staging -> H2D -> `lsd_forward` (all of its streams) -> D2H.  Same kernels, same
        numerics as the launch-by-launch path (tests compare them bitwise)."""
        m = self.model
        dev = self.device
        v = np.stack(visuals)
        a = np.stack(audios)
        dt = torch.float16 if self.use_half_precision else torch.float32
        with m._lsd_lock:
            key = (v.shape, a.shape, dt, m.state_generation())
            ent = self._graphs.get(key)
            if ent is None:
                for k in [k for k in self._graphs if k[3] != key[3]]:      # stale generations
                    del self._graphs[k]
                ent = self._graphs[key] = self._capture_graph(v.shape, a.shape, dt)
                self.graph_captures += 1
            vh, ah, oh, graph = ent["vh"], ent["ah"], ent["oh"], ent["graph"]
            vh.copy_(torch.from_numpy(v))
            ah.copy_(torch.from_numpy(a))
            graph.replay()
            torch.cuda.current_stream(dev).synchronize()
            return [float(x) for x in oh.tolist()]

    def _capture_graph(self, vshape, ashape, dt):
        m = self.model
        dev = self.device
        B, _, T, H, W = vshape
        F_, Ta = ashape[2], ashape[3]
        ent = {
            "vh": torch.empty(vshape, dtype=dt).pin_memory(), "ah": torch.empty(ashape, dtype=dt).pin_memory(),
            "vd": torch.empty(vshape, dtype=dt, device=dev), "ad": torch.empty(ashape, dtype=dt, device=dev),
            "od": torch.empty(B, dtype=torch.float32, device=dev), "oh": torch.empty(B, dtype=torch.float32).pin_memory(),
            "ws": torch.empty(m.workspace_bytes(B, T, H, W, F_, Ta) + 1024, dtype=torch.uint8, device=dev),   # private: its padding persists
        }
        ent["vh"].zero_()
        ent["ah"].zero_()

        def body():
            ent["vd"].copy_(ent["vh"], non_blocking=True)
            ent["ad"].copy_(ent["ah"], non_blocking=True)
            m.forward_into(ent["vd"], ent["ad"], ent["od"], ent["ws"])
            ent["oh"].copy_(ent["od"], non_blocking=True)

        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(2):       # the first call of a shape uploads stage programs and zeroes the padding: not capturable
                body()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            body()
        ent["graph"] = g
        return ent

    def score_batches(self, batches) -> List[torch.Tensor]:
        """Pipelined scoring of a sequence of HOST batches `(visual (B,3,T,H,W), audio (B,1,F,Ta))` (torch CPU tensors, ideally
        pinned): the H2D copies of the next batches run on a copy stream while batch k is scored, logits come back through
        pinned memory.  Returns one fp32 CPU tensor of logits per batch.  Same numerics as calling the model batch by batch."""
        with self.model._lsd_lock:      # the cached device slots make this call non-re-entrant; serialise like forward()
            return self._score_batches_locked(batches)

    def _score_batches_locked(self, batches) -> List[torch.Tensor]:
        dev = self.device
        m = self.model
        comp = torch.cuda.current_stream(dev)
        copy = getattr(self, "_copy_stream", None)
        if copy is None:
            copy = self._copy_stream = torch.cuda.Stream(dev)
        # three device slots: the copy stream stays busy back to back (copy and forward take about the same time at B=64 —
        # 4.1 ms of PCIe vs 3.9 ms of compute — so two slots leave bubbles whenever either one jitters)
        NS = 3
        if getattr(self, "_slot_cache", None) is None:      # device slots and events are kept across calls
            self._slot_cache = ([None] * NS, [torch.cuda.Event() for _ in range(NS)], [torch.cuda.Event() for _ in range(NS)])
        slots, ready, free = self._slot_cache
        outs: List[torch.Tensor] = []
        pool, pool_off = None, 0
        stage = getattr(self, "_u8_stage", None)
        if stage is None:
            stage = self._u8_stage = [None] * NS
        L = _cabi.lib()
        state = {"mode": "fp32" if self.use_half_precision else self.host_transport}
        if state["mode"] == "auto" and getattr(self, "_auto_prefers_fp32", False):
            state["mode"] = "fp32"       # an earlier call on this predictor measured the pack slower than the copy (busy host / several GPUs)

        def split_count(B):
            """Windows of a batch that cross PCIe as fp32 while the host threads pack the rest (split transport): a batch costs the
            pipeline max(PCIe time, pack time), so the fp32 share f equalises  f*t32 + (1-f)*t32/4  and  (1-f)*T + 0.33 ms  (t32: the
            fp32 bytes of the whole batch at ~52 GB/s, T: the measured pack time of a whole batch).  0 until a pack has been measured."""
            if not self.host_split or B < 2:
                return 0
            if isinstance(self.host_split, float):
                return int(round(self.host_split * B))
            return int(round(getattr(self, "_split_frac", 0.0) * B)) if B >= 8 else 0

        def start(k, vh, ah):
            """Host side of batch k, first half: starts the uint8 pack on the library's host threads (the call returns at once;
            this thread goes on to enqueue batch k-1).  No Python helper thread: a second Python thread that makes CUDA calls was
            measured to slow every later single-window call of the process by ~1 ms."""
            s = k % NS
            if self.use_half_precision:
                vh, ah = vh.half(), ah.half()
            if state["mode"] != "fp32" and vh.dtype == torch.float32 and vh.device.type == "cpu" and vh.is_contiguous() and vh.numel() > 0:
                fresh = stage[s] is None or stage[s].shape != vh.shape
                if fresh:
                    stage[s] = torch.empty(vh.shape, dtype=torch.uint8).pin_memory()
                elif k >= NS:
                    ready[s].synchronize()    # the H2D copy that last read this staging buffer (batch k - NS) has finished
                B = int(vh.shape[0])
                wbytes = vh[0].numel()
                na = min(split_count(B), B - 1) if wbytes % 16 == 0 else 0       # (lsd_expand_u8 works in 16-byte pieces)
                if L.lsd_host_pack_u8_begin(vh.data_ptr() + 4 * na * wbytes, stage[s].data_ptr(), (B - na) * wbytes, self.host_pack_threads) == _cabi.LSD_OK:
                    return (k, vh, ah, s, fresh, na)
            return (k, vh, ah, None, False, 0)

        def finish(st):
            """-> (video to ship, audio, transport label, na): na > 0 = split transport (video is then (fp32 windows, packed rest))."""
            k, vh, ah, s, fresh, na = st
            if s is None:
                return vh, ah, "fp32", 0
            ok = L.lsd_host_pack_u8_end()
            if state["mode"] == "fp32":          # the transport was given up while this batch's pack was queued: drained, shipped as fp32
                return vh, ah, "fp32", 0
            if ok == 1:
                B = int(vh.shape[0])
                d = self.__dict__
                first_ever = d.setdefault("_pack_jobs_seen", 0) == 0     # the very first pack of this predictor also starts the pack threads
                d["_pack_jobs_seen"] += 1
                T_ms = L.lsd_host_pack_last_ms() * B / max(1, B - na)     # pack time of a whole batch, from this (possibly partial) pack
                t32 = vh.numel() * 4 / 52e9                               # the fp32 bytes at ~52 GB/s of PCIe gen5 x16
                steady = k >= 1 and not fresh      # not the first batch of a call, not the first pack into a freshly pinned staging buffer
                if steady and self.host_split:
                    f = (T_ms * 1e-3 + 0.33e-3 - t32 / 4) / (0.75 * t32 + T_ms * 1e-3)
                    f = min(0.6, max(0.0, f))
                    if f < 0.05:
                        f = 0.0
                    self._split_frac = f if not hasattr(self, "_split_frac") else 0.5 * self._split_frac + 0.5 * f
                if state["mode"] == "auto" and not self.host_split:
                    # "auto" stops packing only when packing is the slower way (auto_transport_gives_up_packing; histories are kept
                    # across calls, so a three-batch warm-up call can decide for the next one).  Measured (AVX-512 loop, non-temporal
                    # stores, queued jobs): 16 host threads for one GPU pack a 64-window batch in 2.2 ms against >= 4.4 ms of copy;
                    # 12 threads per GPU with two GPUs packing at once need 3.3 ms (4.3 - 4.7 ms per step for the fp32 copy there);
                    # eight GPUs fed at once: ~12 ms per pack whatever the thread count against 6.5 - 9.8 ms per step for the copy —
                    # the pack moves more host-DRAM bytes than the copy it saves, and there the host memory, not PCIe, is the limit.
                    every, recent = d.setdefault("_pack_ms_all", []), d.setdefault("_pack_ms_hist", [])
                    if not first_ever:
                        every.append(T_ms)
                        del every[:-8]
                    if steady:
                        recent.append(T_ms)
                        del recent[:-8]
                    if auto_transport_gives_up_packing(recent, every, t32):
                        state["mode"] = "fp32"             # this batch is packed and exact: it still ships packed, the next ones as fp32
                        self._auto_prefers_fp32 = True     # remembered for the later calls of this predictor
                if na > 0:
                    return (vh, stage[s]), ah, "u8 + fp32 split (host-packed part exact)", na
                return stage[s], ah, "u8 (host-packed, exact)", 0
            state["mode"] = "fp32"               # not k/255 data: stop checking for the rest of this call
            return vh, ah, "fp32", 0

        it = iter(batches)
        pend = []                       # host side started, not yet shipped: batches k, k+1 (the library queues two pack jobs)
        started = [0]

        def fill():
            while len(pend) < 2:
                nxt = next(it, None)
                if nxt is None:
                    return
                pend.append(start(started[0], *nxt))
                started[0] += 1

        fill()
        k = 0
        split_slots = getattr(self, "_split_slots", None)
        if split_slots is None:
            split_slots = self._split_slots = [None] * NS
        try:
            while pend:
                vh, ah, transport, na = finish(pend.pop(0))                     # batch k is packed (or goes as it is)
                fill()          # batch k+1 is being packed while batch k is enqueued, the pack of batch k+2 is queued behind it
                s = k % NS
                self.last_transport = transport        # of the last batch shipped
                if na > 0:
                    # split transport: windows [0, na) cross PCIe as fp32, the rest packed; the packed part is expanded next to the
                    # fp32 part on the device (lsd_expand_u8: the reference's own astype(float32) / 255.0, bit for bit) and ONE fp32
                    # batch is scored
                    v32, v8 = vh
                    B = int(v32.shape[0])
                    wbytes = v32[0].numel()
                    self.last_h2d_bytes_per_batch = 4 * na * wbytes + (B - na) * wbytes + ah.numel() * ah.element_size()
                    ss = split_slots[s]
                    if ss is None or ss[0].shape != v32.shape or ss[2].shape != ah.shape:
                        ss = split_slots[s] = (torch.empty(v32.shape, dtype=torch.float32, device=dev), torch.empty(v32.shape, dtype=torch.uint8, device=dev),
                                               torch.empty(ah.shape, dtype=ah.dtype, device=dev))
                        free[s].record(comp)
                    with torch.cuda.stream(copy):
                        copy.wait_event(free[s])          # the forward that last read this slot has finished
                        ss[0][:na].copy_(v32[:na], non_blocking=True)
                        ss[1][:B - na].copy_(v8[:B - na], non_blocking=True)
                        ss[2].copy_(ah, non_blocking=True)
                        ready[s].record(copy)
                    comp.wait_event(ready[s])
                    rc = L.lsd_expand_u8(ss[1].data_ptr(), ss[0].data_ptr() + 4 * na * wbytes, (B - na) * wbytes, comp.cuda_stream)
                    if rc != _cabi.LSD_OK:
                        raise RuntimeError(f"lsd_expand_u8 failed ({rc})")
                    logits = m(ss[0], ss[2])
                else:
                    self.last_h2d_bytes_per_batch = vh.numel() * vh.element_size() + ah.numel() * ah.element_size()
                    if slots[s] is None or slots[s][0].shape != vh.shape or slots[s][0].dtype != vh.dtype or slots[s][1].shape != ah.shape:
                        slots[s] = (torch.empty(vh.shape, dtype=vh.dtype, device=dev), torch.empty(ah.shape, dtype=ah.dtype, device=dev))
                        free[s].record(comp)
                    with torch.cuda.stream(copy):
                        copy.wait_event(free[s])          # the forward that last read this slot has finished
                        slots[s][0].copy_(vh, non_blocking=True)
                        slots[s][1].copy_(ah, non_blocking=True)
                        ready[s].record(copy)
                    comp.wait_event(ready[s])
                    logits = m(slots[s][0], slots[s][1])
                free[s].record(comp)
                # logits come back through one pinned block per 256 batches (a pinned allocation per step costs ~0.1-0.4 ms)
                nb = int(logits.numel())
                if pool is None or pool_off + nb > pool.numel():
                    pool = torch.empty(max(256 * nb, 4096), dtype=torch.float32, pin_memory=True)
                    pool_off = 0
                host = pool[pool_off:pool_off + nb].view(logits.shape)
                pool_off += nb
                host.copy_(logits.float(), non_blocking=True)
                outs.append(host)
                k += 1
        except BaseException:
            for st in pend:
                if st[3] is not None:
                    L.lsd_host_pack_u8_end()     # never leave a pack job in flight behind an error
            raise
        comp.synchronize()
        return outs

    def _infer_confidences(self, visuals: Sequence[np.ndarray], audios: Sequence[np.ndarray]) -> List[float]:
        return [self._calibrate(l) for l in self._infer_logits(visuals, audios)]

    def _infer_confidence(self, visual_np: np.ndarray, audio_np: np.ndarray) -> float:
        """Run a single forward pass, apply output calibration, return P(REAL)."""
        return self._infer_confidences([visual_np], [audio_np])[0]

    # ------------------------------------------------------------------ aggregation helpers (host numpy, as the reference)
    def _robust_confidence(self, confidences: List[float]) -> float:
        """predictor.py:246-260 (single implementation: `lipsync_b200.aggregate._robust`)."""
        return _agg._robust(confidences, self.confidence_smoothing, self.trim_ratio)

    def _speech_weighted_confidence(self, confidences: List[float], speaking_scores: List[float],
                                    vad_weights: Optional[List[float]] = None) -> float:
        """predictor.py:262-293 (single implementation: `lipsync_b200.aggregate._speech_weighted`)."""
        return _agg._speech_weighted(confidences, speaking_scores, vad_weights, self.confidence_smoothing, self.trim_ratio)

    @staticmethod
    def _smoothing_windows(t_v: int, t_a: int) -> Tuple[List[Tuple[int, int, int, int]], List[Tuple[int, int]]]:
        """Window spans of `_temporal_smoothed_confidence` (predictor.py:302-325): (v0, v1, a0, a1) + reported spans."""
        wins = [(0, t_v, 0, t_a)]
        spans = [(0, max(1, t_v))]
        win_v = max(12, t_v // 2)
        win_a = max(48, t_a // 2)
        if t_v >= win_v and t_a >= win_a:
            v_starts = [0, max(0, (t_v - win_v) // 2), max(0, t_v - win_v)]
            for v_start in v_starts:
                v_end = min(t_v, v_start + win_v)
                a_start = int(round(v_start * (t_a / max(1, t_v))))
                a_end = min(t_a, a_start + win_a)
                if (v_end - v_start) >= 16 and (a_end - a_start) >= 64:
                    wins.append((v_start, v_end, a_start, a_end))
                    spans.append((v_start, v_end))
        return wins, spans

    def _temporal_smoothed_confidence(self, visual_np: np.ndarray, audio_np: np.ndarray):
        t_v = int(visual_np.shape[1])
        t_a = int(audio_np.shape[2])
        wins, spans = self._smoothing_windows(t_v, t_a)
        confidences: List[float] = []
        # full window and the half windows have different shapes: one batch per distinct shape, order preserved
        by_shape = {}
        for i, (v0, v1, a0, a1) in enumerate(wins):
            by_shape.setdefault((v1 - v0, a1 - a0), []).append(i)
        res = [0.0] * len(wins)
        for idxs in by_shape.values():
            vs = [np.ascontiguousarray(visual_np[:, wins[i][0]:wins[i][1]]) for i in idxs]
            as_ = [np.ascontiguousarray(audio_np[:, :, wins[i][2]:wins[i][3]]) for i in idxs]
            for i, c in zip(idxs, self._infer_confidences(vs, as_)):
                res[i] = c
        confidences = res
        return self._robust_confidence(confidences), confidences, spans

    @staticmethod
    def _audio_start(v_start: int, total_a: int, total_v_frames: int, chunk_a_size: int = 128) -> int:
        a_ratio = total_a / max(1, total_v_frames)
        a_start = int(round(v_start * a_ratio))
        if a_start + chunk_a_size > total_a:
            a_start = max(0, total_a - chunk_a_size)
        return a_start

    def _align_audio_chunk(self, audio_np_full: np.ndarray, v_start: int, total_v_frames: int, chunk_a_size: int = 128) -> np.ndarray:
        total_a = int(audio_np_full.shape[2])
        a_start = self._audio_start(v_start, total_a, total_v_frames, chunk_a_size)
        a_end = min(total_a, a_start + chunk_a_size)
        chunk = audio_np_full[:, :, a_start:a_end]
        if chunk.shape[2] < chunk_a_size:
            pad = np.repeat(chunk[:, :, -1:], chunk_a_size - chunk.shape[2], axis=2)
            chunk = np.concatenate([chunk, pad], axis=2)
        return chunk

    def _run_chunked_inference(self, chunks: List[np.ndarray], chunk_starts: List[int], audio_np_full: np.ndarray,
                               total_v_frames: int) -> Tuple[float, List[float]]:
        """Score every chunk of a track (batched) and aggregate; returns (aggregated_confidence, per_chunk_confidences)."""
        audios = [self._align_audio_chunk(audio_np_full, v_start, total_v_frames) for v_start in chunk_starts]
        chunk_confs = self._infer_confidences(list(chunks), audios) if len(chunks) else []
        return self._robust_confidence(chunk_confs), chunk_confs

    # ------------------------------------------------------------------ device-side window builder (SURVEY.md §8f-1)
    def score_track_logits(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                           chunk_a_size: int = 128, audio_starts_from: Optional[Sequence[int]] = None) -> torch.Tensor:
        """uint8 track `(n_frames,H,W,3)` + window start frames + clip log-mel `(1,F,Ta_full)` (both on the device)
        -> fp32 logits `(n_windows,)` on the device.  Windows are built on the GPU (`/255`, audio alignment).
        `audio_starts_from`: absolute start frames used for the audio alignment when `track_u8` is only a rank-local span
        of the full track and `starts` are relative to that span (sharded long videos)."""
        return self._score_windows(track_u8, starts, mel_full, total_v_frames, chunk_a_size, audio_starts_from, False)[0]

    def _score_windows(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                       chunk_a_size: int, audio_starts_from: Optional[Sequence[int]], with_feats: bool):
        """`score_track_logits`, and with `with_feats` also the head's input rows (`lsd_score_branch_features`): (logits, feats)."""
        m = self.model
        dev = m._device()
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        n = len(starts)
        logits = torch.empty(n, dtype=torch.float32, device=dev)
        feats = torch.empty((n, _cabi.LSD_BRANCH_FEATURES), dtype=torch.float32, device=dev) if with_feats else None
        if n == 0:
            return logits, feats
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n)
            need = L.lsd_score_workspace_bytes(h.ptr, batch, self.chunk_size, H, W, F_, chunk_a_size, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            if n > batch and prec == _cabi.LSD_PREC_BF16:
                need = 2 * need      # a double workspace lets lsd_score_windows overlap the tail of batch k with the encoder of batch k+1
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                if len(audio_starts_from) != n:
                    raise ValueError("audio_starts_from must have one entry per window")
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), chunk_a_size) for v in audio_starts_from])
            stream = torch.cuda.current_stream(dev).cuda_stream
            if with_feats:
                rc = L.lsd_score_branch_features(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, self.chunk_size,
                                                 mel_full.data_ptr(), F_, Ta_full, int(total_v_frames), chunk_a_size, prec, batch,
                                                 logits.data_ptr(), feats.data_ptr(), ws.data_ptr(), ws.numel(), stream)
            else:
                rc = L.lsd_score_windows(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, self.chunk_size, mel_full.data_ptr(),
                                         F_, Ta_full, int(total_v_frames), chunk_a_size, prec, batch, logits.data_ptr(),
                                         ws.data_ptr(), ws.numel(), stream)
            _cabi.check(h.ptr, rc)
        return logits, feats

    # ------------------------------------------------------------------ branch attribution (lsd_score_branch_features, lsd_branch_attribution)
    BRANCHES = _agg.BRANCHES
    #: windows of the track background: at most this many, spread evenly over the track
    TRACK_BACKGROUND_MAX = 64

    def score_track_branch_features(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                                    audio_starts_from: Optional[Sequence[int]] = None, chunk_a_size: int = 128):
        """`score_track_logits` that also returns every window's head input row: `(logits (n,), feats (n, 448))` fp32 on the
        device.  feats row i is [cls 256 | raw 64 | delta 64 | hf 64], what the artifact fusion MLP and the head read for window i;
        the logits are bit for bit those of `score_track_logits`.  Both precisions."""
        return self._score_windows(track_u8, starts, mel_full, total_v_frames, chunk_a_size, audio_starts_from, True)

    @staticmethod
    def track_background_index(n: int, max_rows: int = 64) -> List[int]:
        """Windows of the track background of an n-window track: M = min(n, max_rows) of them, (arange(M) * n) // M."""
        M = min(int(n), int(max_rows))
        return [(k * int(n)) // M for k in range(M)]

    def branch_attribution(self, feats: torch.Tensor, background: torch.Tensor):
        """Exact Shapley values of the head's four inputs (`lsd_branch_attribution`).  `feats`: (n, 448) head input rows
        (`score_track_branch_features`); `background`: (M, 448) rows, 1 <= M <= 256, on the same device, fp32.  Returns
        `(values (n, 16), phi (n, 4))` fp32 on the device: values[i, S] = v_i(S), the mean over the background rows j of the head's
        logit on the row that takes branch p (sync, raw, delta, hf = bit p of S) from window i when bit p is set and from row j
        otherwise; values[i, 15] is window i's own logit.  phi[i, p] is branch p's Shapley value; the four sum to
        values[i, 15] - values[i, 0]."""
        want = self.model._device() if self.model is not None else self.device
        for name, t in (("feats", feats), ("background", background)):
            if not isinstance(t, torch.Tensor) or t.dim() != 2 or t.shape[1] != _cabi.LSD_BRANCH_FEATURES:
                raise ValueError(f"{name} must be a ({'n' if name == 'feats' else 'M'}, {_cabi.LSD_BRANCH_FEATURES}) tensor, got "
                                 f"{tuple(t.shape) if isinstance(t, torch.Tensor) else type(t).__name__}")
            if t.dtype != torch.float32:
                raise ValueError(f"{name} must be float32, got {t.dtype}")
            if t.device != want:
                raise ValueError(f"{name} is on {t.device}, the model on {want}")
        M = int(background.shape[0])
        if not 1 <= M <= _cabi.LSD_MAX_BACKGROUND:
            raise ValueError(f"{M} background rows: expected 1 to {_cabi.LSD_MAX_BACKGROUND}")
        n = int(feats.shape[0])
        if n * (15 * M + 1) > 2 ** 31 - 1:
            raise ValueError(f"{n} windows x {M} background rows: too many coalition rows for one call")
        if want.type != "cuda" or self.model is None:
            raise ValueError(f"branch attribution runs on a CUDA model, the predictor is on {want}")
        m = self.model
        dev = m._device()
        values = torch.empty((n, 16), dtype=torch.float32, device=dev)
        phi = torch.empty((n, _cabi.LSD_BRANCHES), dtype=torch.float32, device=dev)
        if n == 0:
            return values, phi
        feats = feats.contiguous()
        background = background.contiguous()
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            need = L.lsd_branch_attribution_workspace_bytes(n, M)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            ws = torch.empty(int(need), dtype=torch.uint8, device=dev)
            rc = L.lsd_branch_attribution(h.ptr, feats.data_ptr(), n, background.data_ptr(), M, values.data_ptr(), phi.data_ptr(),
                                          ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return values, phi

    def attribution_track(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                          background="track", confidence_threshold: float = 0.5,
                          audio_starts_from: Optional[Sequence[int]] = None) -> Dict[str, Any]:
        """Branch attribution of a track's windows: was a window called fake because lips and speech disagree (sync) or because
        the pixels carry generator artifacts (raw, delta: the temporal-inconsistency detector; hf: the high-frequency detector)?
        One `score_track_branch_features` call, then `branch_attribution` against `background`: "track" (the track's own windows,
        `track_background_index`: what sets a window apart from the rest of the clip) or an (M, 448) tensor of feature rows, e.g.
        those of windows known to be real ("reference").  Returns host arrays:
          `branches`; `logits` (n,); `values` (n, 16); `phi` (n, 4); `base_logit` (n,) = values[:, 0], the background's expected
          logit; `background` ("track" or "reference") and `background_size` (M);
          the `aggregate.branch_attribution_summary` of phi and the calibrated P(real) at `confidence_threshold`, its timeline in
          the frames of `window_starts`;
          `window_starts`: the windows' first frames (those of `audio_starts_from` when given: absolute video frames).
        It reports only: nothing here enters a verdict."""
        n = len(starts)
        if isinstance(background, str) and background != "track":
            raise ValueError(f"background must be 'track' or an (M, {_cabi.LSD_BRANCH_FEATURES}) tensor, got {background!r}")
        if isinstance(background, str) and n == 0:
            raise ValueError("a track background needs at least one window")
        logits, feats = self.score_track_branch_features(track_u8, starts, mel_full, total_v_frames, audio_starts_from=audio_starts_from)
        if isinstance(background, str):
            idx = torch.tensor(self.track_background_index(n, self.TRACK_BACKGROUND_MAX), dtype=torch.long, device=feats.device)
            bg, kind = feats.index_select(0, idx), "track"
        else:
            bg, kind = background, "reference"
        values, phi = self.branch_attribution(feats, bg)
        lg = logits.cpu().numpy()
        vals = values.cpu().numpy()
        ph = phi.cpu().numpy()
        probs = np.array([self._calibrate(float(x)) for x in lg.tolist()], dtype=np.float64)
        window_starts = [int(s) for s in (audio_starts_from if audio_starts_from is not None else starts)]
        res = {"branches": list(self.BRANCHES), "logits": lg, "values": vals, "phi": ph, "base_logit": vals[:, 0],
               "background": kind, "background_size": int(bg.shape[0])}
        res.update(_agg.branch_attribution_summary(ph, probs, confidence_threshold, self.confidence_smoothing, self.trim_ratio,
                                                   starts=window_starts, T=self.chunk_size))
        res["window_starts"] = window_starts
        return res

    def score_track_offsets(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                            offsets: Sequence[int], chunk_a_size: int = 128, audio_starts_from: Optional[Sequence[int]] = None):
        """`score_track_logits` with K audio offsets per window (`lsd_score_offsets`): offset d (mel columns, 10 ms, d > 0 =
        audio later) moves the window's aligned audio start a_i to clamp(a_i + d), clamped like `_audio_start`.  The video side of
        a window is computed once for all offsets.  Returns `(logits (n,K) fp32 on the device, effective audio starts (n,K)
        np.int32, valid (n,K) bool)`; (i, k) is valid when 0 <= a_i + d_k <= T_full - chunk_a_size (no clamping)."""
        m = self.model
        dev = m._device()
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        offs = [int(d) for d in offsets]
        K = len(offs)
        if not 1 <= K <= _cabi.LSD_MAX_AUDIO_VARIANTS:
            raise ValueError(f"{K} offsets: expected 1 to {_cabi.LSD_MAX_AUDIO_VARIANTS}")
        n = len(starts)
        if audio_starts_from is not None and len(audio_starts_from) != n:
            raise ValueError("audio_starts_from must have one entry per window")
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        base = np.array([self._audio_start(int(v), Ta_full, int(total_v_frames), chunk_a_size)
                         for v in (audio_starts_from if audio_starts_from is not None else starts)], dtype=np.int64).reshape(n, 1)
        moved = base + np.asarray(offs, dtype=np.int64).reshape(1, K)
        valid = (moved >= 0) & (moved <= Ta_full - chunk_a_size)
        logits = torch.empty(n, K, dtype=torch.float32, device=dev)
        eff = np.zeros((n, K), dtype=np.int32)
        if n == 0:
            return logits, eff, valid
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n)
            need = L.lsd_score_offsets_workspace_bytes(h.ptr, batch, K, self.chunk_size, H, W, F_, chunk_a_size, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None if audio_starts_from is None else (C.c_int32 * n)(*[int(a) for a in base[:, 0]])
            offs_c = (C.c_int32 * K)(*offs)
            eff_c = (C.c_int32 * (n * K))()
            rc = L.lsd_score_offsets(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, self.chunk_size, mel_full.data_ptr(), F_, Ta_full,
                                     int(total_v_frames), chunk_a_size, offs_c, K, prec, batch, logits.data_ptr(), eff_c,
                                     ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        eff[:] = np.frombuffer(eff_c, dtype=np.int32).reshape(n, K)
        return logits, eff, valid

    @staticmethod
    def default_av_offsets(Ta_full: int, total_v_frames: int, max_frames: int = 7) -> Tuple[List[int], List[int]]:
        """Whole video frames -max_frames..+max_frames and their offsets in mel columns, converted with the ratio `_audio_start`
        uses (round(f * T_full / total_v_frames), round-half-even)."""
        frames = list(range(-int(max_frames), int(max_frames) + 1))
        a_ratio = Ta_full / max(1, total_v_frames)
        return frames, [int(round(f * a_ratio)) for f in frames]

    def estimate_av_offset(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                           offsets: Optional[Sequence[int]] = None, chunk_a_size: int = 128,
                           audio_starts_from: Optional[Sequence[int]] = None) -> Dict[str, Any]:
        """Audio-visual offset of a track: `score_track_offsets` + `aggregate.av_offset_profile` on the calibrated confidences,
        aggregated like the window confidences (`confidence_smoothing`, `trim_ratio`).  Default offsets: whole video frames
        -7..+7 (`default_av_offsets`).  Offsets are also reported in seconds (one mel column = 10 ms).  Reporting only: the
        offset changes no verdict."""
        Ta_full = int(mel_full.shape[2])
        frames = None
        if offsets is None:
            frames, offsets = self.default_av_offsets(Ta_full, total_v_frames)
        offsets = [int(d) for d in offsets]
        logits, _, valid = self.score_track_offsets(track_u8, starts, mel_full, total_v_frames, offsets, chunk_a_size, audio_starts_from)
        confs = np.array([self._calibrate(float(x)) for x in logits.cpu().flatten().tolist()], dtype=np.float32).reshape(valid.shape)
        res = _agg.av_offset_profile(confs, valid, offsets, self.confidence_smoothing, self.trim_ratio)
        res["offsets_sec"] = [d * _MEL_HOP_SEC for d in offsets]
        res["best_offset_sec"] = res["best_offset"] * _MEL_HOP_SEC if res["best_offset"] is not None else None
        if frames is not None:
            res["offset_frames"] = frames
        return res

    # ------------------------------------------------------------------ occlusion evidence (lsd_score_occlusions)
    def score_track_occlusions(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                               boxes, fill: int = 128, chunk_a_size: int = 128,
                               audio_starts_from: Optional[Sequence[int]] = None) -> torch.Tensor:
        """`score_track_logits` with K occlusion boxes per window (`lsd_score_occlusions`).  `boxes`: a `(K, 7)` int array or a
        sequence of 7-tuples `(t0, t1, y0, y1, x0, x1, src)` in window coordinates; pixels of frames [t0,t1) x rows [y0,y1) x columns
        [x0,x1) are replaced by frame `src` of the un-occluded window (src >= 0) or by `fill` (src = -1).  An empty box leaves the
        window as it is.  The occluded windows are built on the device.  Returns fp32 logits `(n, K)` on the device; entry (i, k)
        is bit for bit the logit of window i occluded by box k, with window i's audio slice."""
        m = self.model
        dev = m._device()
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T = self.chunk_size
        bx = np.asarray(boxes, dtype=np.int64)
        if bx.ndim != 2 or bx.shape[1] != 7:
            raise ValueError(f"boxes must be (K, 7) (t0, t1, y0, y1, x0, x1, src), got shape {bx.shape}")
        K = int(bx.shape[0])
        if not 1 <= K <= _cabi.LSD_MAX_OCCLUSIONS:
            raise ValueError(f"{K} occlusion boxes: expected 1 to {_cabi.LSD_MAX_OCCLUSIONS}")
        for k, (t0, t1, y0, y1, x0, x1, src) in enumerate(bx.tolist()):
            if not (0 <= t0 <= t1 <= T and 0 <= y0 <= y1 <= H and 0 <= x0 <= x1 <= W):
                raise ValueError(f"box {k} {bx[k].tolist()} is not inside the {T}x{H}x{W} window")
            if not -1 <= src < T:
                raise ValueError(f"box {k}: src {src} is outside -1..{T - 1}")
        if not 0 <= int(fill) <= 255:
            raise ValueError(f"fill must be a uint8 value, got {fill}")
        n = len(starts)
        if audio_starts_from is not None and len(audio_starts_from) != n:
            raise ValueError("audio_starts_from must have one entry per window")
        for i, s in enumerate(starts):
            if not 0 <= int(s) <= n_frames - T:
                raise ValueError(f"window {i} [{int(s)},{int(s) + T}) is outside the {n_frames}-frame track")
        logits = torch.empty(n, K, dtype=torch.float32, device=dev)
        if n == 0:
            return logits
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n * K)
            need = L.lsd_score_occlusions_workspace_bytes(h.ptr, batch, T, H, W, F_, chunk_a_size, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            if n * K > batch and prec == _cabi.LSD_PREC_BF16:
                need = 2 * need      # a double workspace lets the batches overlap as in score_track_logits
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), chunk_a_size) for v in audio_starts_from])
            boxes_c = (_cabi.LsdOcclusion * K)(*[_cabi.LsdOcclusion(*row) for row in bx.tolist()])
            rc = L.lsd_score_occlusions(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, T, mel_full.data_ptr(), F_, Ta_full,
                                        int(total_v_frames), chunk_a_size, boxes_c, K, int(fill), prec, batch, logits.data_ptr(),
                                        ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return logits

    @staticmethod
    def freeze_segment_boxes(T: int, segment_frames: int, H: int = 96, W: int = 96) -> List[Tuple[int, ...]]:
        """Freeze boxes: segment j = frames [j*s, min((j+1)*s, T)) replaced, over the whole H x W frame, by the frame just before
        it (the frame just after it for the first segment).  It asks: what if the mouth stopped moving here?"""
        T, s = int(T), int(segment_frames)
        if s < 1:
            raise ValueError(f"segment_frames must be >= 1, got {segment_frames}")
        if s >= T:
            raise ValueError(f"a segment of {s} frames covers the whole {T}-frame window: there is no frame to freeze to")
        out = []
        for t0 in range(0, T, s):
            t1 = min(t0 + s, T)
            out.append((t0, t1, 0, int(H), 0, int(W), t0 - 1 if t0 > 0 else t1))
        return out

    @staticmethod
    def fill_cell_boxes(T: int, H: int, W: int, grid: int) -> List[Tuple[int, ...]]:
        """Fill boxes: the crop cut into grid x grid cells (edges round(j*H/grid), round(j*W/grid)), row-major, each cell filled
        over all T frames with the call's fill value."""
        g = int(grid)
        if not 1 <= g <= min(int(H), int(W)):
            raise ValueError(f"grid must be in 1..{min(int(H), int(W))}, got {grid}")
        ye = [int(round(j * H / g)) for j in range(g + 1)]
        xe = [int(round(j * W / g)) for j in range(g + 1)]
        return [(0, int(T), ye[a], ye[a + 1], xe[b], xe[b + 1], -1) for a in range(g) for b in range(g)]

    def explain_track(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                      segment_frames: int = 4, grid: int = 4, fill: int = 128,
                      audio_starts_from: Optional[Sequence[int]] = None) -> Dict[str, Any]:
        """Occlusion evidence of every window of a track: one `score_track_occlusions` call with an empty box, the freeze segments
        (`freeze_segment_boxes`) and the fill cells (`fill_cell_boxes`), K = 1 + 8 + 16 = 25 at the defaults.
        Returns calibrated values:
          `confidence` (n,): P(real) of the plain window;
          `temporal` (n, S), `spatial` (n, grid, grid): P(real) with the region hidden MINUS `confidence`.  A value > 0 means
            hiding the region made the window look more real: the region carried evidence of a fake.  A value < 0: it carried
            evidence of a real video;
          `spatial_mean` (grid, grid): `spatial` averaged over the windows;
          `frame_first`, `frame_evidence`: the per-frame timeline of `temporal` (`aggregate.frame_evidence_timeline`), in the
            frame numbers of `audio_starts_from` when given (absolute video frames), otherwise of `starts`;
          `segment_frames`, `grid`, `fill`."""
        T = self.chunk_size
        H, W = int(track_u8.shape[1]), int(track_u8.shape[2])
        freeze = self.freeze_segment_boxes(T, segment_frames, H, W)
        cells = self.fill_cell_boxes(T, H, W, grid)
        boxes = [(0, 0, 0, 0, 0, 0, -1)] + freeze + cells
        logits = self.score_track_occlusions(track_u8, starts, mel_full, total_v_frames, boxes, fill=fill, audio_starts_from=audio_starts_from)
        n, S, g = len(starts), len(freeze), int(grid)
        probs = np.array([self._calibrate(float(x)) for x in logits.cpu().flatten().tolist()], dtype=np.float64).reshape(n, len(boxes))
        conf = probs[:, 0]
        temporal = probs[:, 1:1 + S] - conf[:, None]
        spatial = (probs[:, 1 + S:] - conf[:, None]).reshape(n, g, g)
        pos = [int(s) for s in (audio_starts_from if audio_starts_from is not None else starts)]
        first, timeline = _agg.frame_evidence_timeline(pos, temporal, int(segment_frames), T)
        return {"confidence": conf, "temporal": temporal, "spatial": spatial,
                "spatial_mean": spatial.mean(axis=0) if n else np.zeros((g, g)),
                "frame_first": first, "frame_evidence": timeline,
                "segment_frames": int(segment_frames), "grid": g, "fill": int(fill)}

    # ------------------------------------------------------------------ audio occlusion evidence (lsd_score_audio_occlusions)
    def score_track_audio_occlusions(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                                     boxes, fill: float = -80.0, chunk_a_size: int = 128,
                                     audio_starts_from: Optional[Sequence[int]] = None) -> torch.Tensor:
        """`score_track_logits` with K audio occlusion boxes per window (`lsd_score_audio_occlusions`).  `boxes`: a `(K, 4)` int
        array or a sequence of 4-tuples `(c0, c1, f0, f1)` in window coordinates; mel columns [c0,c1) x bins [f0,f1) of the window's
        `(F, chunk_a_size)` log-mel slice (`_align_audio_chunk`, after its padding) are set to `fill`.  The default -80 is the floor
        of the library's log-mel (`power_to_db(ref=max, top_db=80)`): silence relative to the clip's maximum.  An empty box leaves
        the slice as it is.  The video side of a window runs once for all its boxes.  Returns fp32 logits `(n, K)` on the device;
        entry (i, k) is bit for bit the logit of window i with its audio slice masked by box k."""
        m = self.model
        dev = m._device()
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        T, Ta = self.chunk_size, int(chunk_a_size)
        bx = np.asarray(boxes, dtype=np.int64)
        if bx.ndim != 2 or bx.shape[1] != 4:
            raise ValueError(f"boxes must be (K, 4) (c0, c1, f0, f1), got shape {bx.shape}")
        K = int(bx.shape[0])
        if not 1 <= K <= _cabi.LSD_MAX_AUDIO_OCCLUSIONS:
            raise ValueError(f"{K} audio occlusion boxes: expected 1 to {_cabi.LSD_MAX_AUDIO_OCCLUSIONS}")
        for k, (c0, c1, f0, f1) in enumerate(bx.tolist()):
            if not (0 <= c0 <= c1 <= Ta and 0 <= f0 <= f1 <= F_):
                raise ValueError(f"audio box {k} {bx[k].tolist()} is not inside the {Ta}-column x {F_}-bin window")
        if not np.isfinite(float(fill)):
            raise ValueError(f"fill must be finite, got {fill}")
        n = len(starts)
        if audio_starts_from is not None and len(audio_starts_from) != n:
            raise ValueError("audio_starts_from must have one entry per window")
        for i, s in enumerate(starts):
            if not 0 <= int(s) <= n_frames - T:
                raise ValueError(f"window {i} [{int(s)},{int(s) + T}) is outside the {n_frames}-frame track")
        logits = torch.empty(n, K, dtype=torch.float32, device=dev)
        if n == 0:
            return logits
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n)
            need = L.lsd_score_audio_occlusions_workspace_bytes(h.ptr, batch, K, T, H, W, F_, Ta, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), Ta) for v in audio_starts_from])
            boxes_c = (_cabi.LsdAudioOcclusion * K)(*[_cabi.LsdAudioOcclusion(*row) for row in bx.tolist()])
            rc = L.lsd_score_audio_occlusions(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, T, mel_full.data_ptr(), F_, Ta_full,
                                              int(total_v_frames), Ta, boxes_c, K, float(fill), prec, batch, logits.data_ptr(),
                                              ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return logits

    @staticmethod
    def mute_segment_boxes(Ta: int, segment_cols: int, F: int = 80) -> List[Tuple[int, ...]]:
        """Mute boxes: segment j = mel columns [j*s, min((j+1)*s, Ta)) of the window's slice, over all F bins.  It asks: what if
        the speech stopped here?  (16 columns = 160 ms.)"""
        Ta, s, F = int(Ta), int(segment_cols), int(F)
        if s < 1 or Ta < 1 or F < 1:
            raise ValueError(f"Ta, segment_cols and F must be >= 1, got {Ta}, {segment_cols} and {F}")
        return [(c0, min(c0 + s, Ta), 0, F) for c0 in range(0, Ta, s)]

    @staticmethod
    def mel_band_boxes(Ta: int, F: int, bands: int) -> List[Tuple[int, ...]]:
        """Band boxes: the F mel bins cut into `bands` bands (edges round(j*F/bands)), low to high, each over all Ta columns."""
        Ta, F, b = int(Ta), int(F), int(bands)
        if Ta < 1:
            raise ValueError(f"Ta must be >= 1, got {Ta}")
        if not 1 <= b <= F:
            raise ValueError(f"bands must be in 1..{F}, got {bands}")
        e = [int(round(j * F / b)) for j in range(b + 1)]
        return [(0, Ta, e[j], e[j + 1]) for j in range(b)]

    def explain_track_audio(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                            segment_cols: int = 16, bands: int = 8, fill: float = -80.0,
                            audio_starts_from: Optional[Sequence[int]] = None) -> Dict[str, Any]:
        """Audio occlusion evidence of every window of a track: one `score_track_audio_occlusions` call with an empty box, the mute
        segments (`mute_segment_boxes`) and the mel bands (`mel_band_boxes`), K = 1 + 8 + 8 = 17 at the defaults (128-column slices).
        Returns calibrated values with the sign convention of `explain_track`:
          `confidence` (n,): P(real) of the plain window (equal to `explain_track`'s);
          `audio_temporal` (n, S), `audio_spectral` (n, bands): P(real) with the box masked MINUS `confidence`.  A value > 0 means
            masking the region made the window look more real: that stretch of speech or band carried evidence of a fake;
          `audio_spectral_mean` (bands,): `audio_spectral` averaged over the windows;
          `column_first`, `column_evidence`: the per-mel-column timeline of `audio_temporal` (`aggregate.frame_evidence_timeline`
            on the windows' audio starts), in absolute clip columns when `audio_starts_from` is given, cut to the clip's columns;
          `frame_first`, `frame_evidence`: that timeline in video frames (`aggregate.columns_to_frames`), to line up with
            `explain_track`'s `frame_evidence`;
          `segment_cols`, `bands`, `band_edges` (bands + 1 mel-bin edges), `fill`."""
        Ta = 128
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        mute = self.mute_segment_boxes(Ta, segment_cols, F_)
        band = self.mel_band_boxes(Ta, F_, bands)
        boxes = [(0, 0, 0, 0)] + mute + band
        logits = self.score_track_audio_occlusions(track_u8, starts, mel_full, total_v_frames, boxes, fill=fill, chunk_a_size=Ta,
                                                   audio_starts_from=audio_starts_from)
        n, S, nb = len(starts), len(mute), int(bands)
        probs = np.array([self._calibrate(float(x)) for x in logits.cpu().flatten().tolist()], dtype=np.float64).reshape(n, len(boxes))
        conf = probs[:, 0]
        temporal = probs[:, 1:1 + S] - conf[:, None]
        spectral = probs[:, 1 + S:] - conf[:, None]
        pos = [self._audio_start(int(s), Ta_full, int(total_v_frames), Ta)
               for s in (audio_starts_from if audio_starts_from is not None else starts)]
        first, cols = _agg.frame_evidence_timeline(pos, temporal, int(segment_cols), Ta)
        cols = cols[:max(0, Ta_full - first)]                             # a slice past the clip's end repeats its last column
        f_first, frames = _agg.columns_to_frames(first, cols, Ta_full, int(total_v_frames))
        return {"confidence": conf, "audio_temporal": temporal, "audio_spectral": spectral,
                "audio_spectral_mean": spectral.mean(axis=0) if n else np.zeros(nb),
                "column_first": first, "column_evidence": cols, "frame_first": f_first, "frame_evidence": frames,
                "segment_cols": int(segment_cols), "bands": nb, "band_edges": [b[2] for b in band] + [band[-1][3]], "fill": float(fill)}

    # ------------------------------------------------------------------ crop-jitter robustness (lsd_score_warps)
    def score_track_warps(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                          warps, chunk_a_size: int = 128, audio_starts_from: Optional[Sequence[int]] = None) -> torch.Tensor:
        """`score_track_logits` with K re-cropped variants per window (`lsd_score_warps`).  `warps`: `(K, 2, 3)` forward affine
        matrices in cv2's convention (src -> dst, as `cv2.warpAffine` takes them), the same for every frame, or `(K, T, 2, 3)`, one
        per frame of the window.  Frame t of variant k is `cv2.warpAffine(frame, M[k, t], (W, H), INTER_LINEAR, BORDER_REPLICATE)`,
        bit for bit, built on the device.  Returns fp32 logits `(n, K)` on the device; entry (i, k) is bit for bit the logit of
        window i re-cropped by variant k, with window i's audio slice."""
        m = self.model
        dev = m._device()
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T = self.chunk_size
        w = self._warp_matrices(warps, T)
        K = int(w.shape[0])
        n = len(starts)
        if audio_starts_from is not None and len(audio_starts_from) != n:
            raise ValueError("audio_starts_from must have one entry per window")
        for i, s in enumerate(starts):
            if not 0 <= int(s) <= n_frames - T:
                raise ValueError(f"window {i} [{int(s)},{int(s) + T}) is outside the {n_frames}-frame track")
        logits = torch.empty(n, K, dtype=torch.float32, device=dev)
        if n == 0:
            return logits
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n * K)
            need = L.lsd_score_warps_workspace_bytes(h.ptr, batch, K, T, H, W, F_, chunk_a_size, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            if n * K > batch and prec == _cabi.LSD_PREC_BF16:
                need = 2 * need      # a double workspace lets the batches overlap as in score_track_logits
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), chunk_a_size) for v in audio_starts_from])
            warps_c = (_cabi.LsdWarp * (K * T)).from_buffer_copy(w.tobytes())
            rc = L.lsd_score_warps(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, T, mel_full.data_ptr(), F_, Ta_full,
                                   int(total_v_frames), chunk_a_size, warps_c, K, prec, batch, logits.data_ptr(), ws.data_ptr(),
                                   ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return logits

    @staticmethod
    def _warp_matrices(warps, T: int) -> np.ndarray:
        """`(K, 2, 3)` or `(K, T, 2, 3)` matrices as a contiguous float64 `(K, T, 2, 3)` array, K checked."""
        w = np.asarray(warps, dtype=np.float64)
        if w.ndim == 3 and w.shape[1:] == (2, 3):
            w = np.broadcast_to(w[:, None], (w.shape[0], T, 2, 3))
        elif not (w.ndim == 4 and w.shape[1:] == (T, 2, 3)):
            raise ValueError(f"warps must be (K, 2, 3) or (K, {T}, 2, 3), got shape {w.shape}")
        if not 1 <= w.shape[0] <= _cabi.LSD_MAX_WARPS:
            raise ValueError(f"{w.shape[0]} warp variants: expected 1 to {_cabi.LSD_MAX_WARPS}")
        return np.ascontiguousarray(w)

    def warp_track_windows(self, track_u8: torch.Tensor, starts: Sequence[int], warps) -> torch.Tensor:
        """The re-cropped windows `score_track_warps` scores, built by the same kernel (`lsd_warp_windows`): uint8
        `(n, K, T, H, W, 3)` on the device, window i under variant k at [i, k].  To look at what a variant does to the crop."""
        m = self.model
        dev = m._device()
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T = self.chunk_size
        w = self._warp_matrices(warps, T)
        K, n = int(w.shape[0]), len(starts)
        for i, s in enumerate(starts):
            if not 0 <= int(s) <= n_frames - T:
                raise ValueError(f"window {i} [{int(s)},{int(s) + T}) is outside the {n_frames}-frame track")
        out = torch.empty((n, K, T, H, W, 3), dtype=torch.uint8, device=dev)
        if n == 0:
            return out
        track_u8 = track_u8.contiguous()
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            need = L.lsd_warp_windows_workspace_bytes(n, K, T, H, W)
            ws = torch.empty(max(int(need), 1), dtype=torch.uint8, device=dev)
            warps_c = (_cabi.LsdWarp * (K * T)).from_buffer_copy(w.tobytes())
            rc = L.lsd_warp_windows(h.ptr, track_u8.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*[int(s) for s in starts]), n, T, warps_c,
                                    K, out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return out

    @staticmethod
    def flip_warp(W: int) -> np.ndarray:
        """Horizontal mirror of a W-pixel-wide crop: x -> W-1-x (cv2.flip(frame, 1) as a warp)."""
        return np.array([[-1.0, 0.0, float(W) - 1.0], [0.0, 1.0, 0.0]])

    @staticmethod
    def shift_scale_rotate_warp(H: int, W: int, dx: float = 0.0, dy: float = 0.0, scale: float = 1.0, angle_deg: float = 0.0) -> np.ndarray:
        """`cv2.getRotationMatrix2D(((W-1)/2, (H-1)/2), angle_deg, scale)` followed by a shift of (dx, dy) pixels: the crop scaled
        by `scale` and turned by `angle_deg` (counter-clockwise, as cv2) about its centre, then moved."""
        a = float(angle_deg) * (np.pi / 180.0)
        alpha, beta = np.cos(a) * float(scale), np.sin(a) * float(scale)
        cx, cy = (float(W) - 1.0) / 2.0, (float(H) - 1.0) / 2.0
        return np.array([[alpha, beta, (1.0 - alpha) * cx - beta * cy + float(dx)],
                         [-beta, alpha, beta * cx + (1.0 - alpha) * cy + float(dy)]])

    @staticmethod
    def jitter_warps(T: int, H: int, W: int, sigma_px: float = 1.5, sigma_scale: float = 0.02, seed: int = 0) -> np.ndarray:
        """(T, 2, 3) per-frame re-crops that model a face tracker's jitter: frame t shifted by (dx_t, dy_t) ~ N(0, sigma_px) and
        scaled about the centre by 1 + s_t, s_t ~ N(0, sigma_scale), all independent (numpy generator seeded with `seed`)."""
        g = np.random.default_rng(int(seed))
        d = g.normal(0.0, float(sigma_px), size=(int(T), 2))
        s = 1.0 + g.normal(0.0, float(sigma_scale), size=int(T))
        return np.stack([Predictor.shift_scale_rotate_warp(H, W, d[t, 0], d[t, 1], s[t]) for t in range(int(T))])

    @staticmethod
    def robustness_variants(T: int, H: int, W: int) -> Tuple[List[str], np.ndarray]:
        """The K = 12 re-crops of `robustness_track`: names and `(K, T, 2, 3)` matrices.  The identity; a horizontal flip; shifts of
        +-4 px in x and in y; scales 0.92 and 1.08; rotations of +-6 degrees; two per-frame tracker jitters (`jitter_warps`,
        sigma 1.5 px and 2 % scale, seeds 0 and 1)."""
        ssr = Predictor.shift_scale_rotate_warp
        fixed = [("identity", ssr(H, W)), ("flip", Predictor.flip_warp(W)),
                 ("shift_x+4", ssr(H, W, dx=4)), ("shift_x-4", ssr(H, W, dx=-4)),
                 ("shift_y+4", ssr(H, W, dy=4)), ("shift_y-4", ssr(H, W, dy=-4)),
                 ("scale_0.92", ssr(H, W, scale=0.92)), ("scale_1.08", ssr(H, W, scale=1.08)),
                 ("rotate+6", ssr(H, W, angle_deg=6)), ("rotate-6", ssr(H, W, angle_deg=-6))]
        mats = [np.broadcast_to(M, (int(T), 2, 3)) for _, M in fixed]
        mats += [Predictor.jitter_warps(T, H, W, 1.5, 0.02, seed) for seed in (0, 1)]
        return [name for name, _ in fixed] + ["jitter_0", "jitter_1"], np.stack(mats)

    def robustness_track(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                         confidence_threshold: float = 0.5, audio_starts_from: Optional[Sequence[int]] = None) -> Dict[str, Any]:
        """Crop-jitter robustness of a track's verdict: one `score_track_warps` call with the K = 12 `robustness_variants`, the
        calibrated P(real) summarised by `aggregate.augmentation_stability`:
          `variants`: the variant names (column order);
          `confidence`: the robust aggregate of the identity column (the plain windows' score);
          `variant_confidence` (K,): the same aggregate per variant;
          `tta_confidence`: the aggregate over windows of the mean P(real) over the variants (flip / shift test-time augmentation);
          `window_spread` (n,): per window, the largest minus the smallest P(real) over the variants;
          `decision_flip_rate`: the fraction of (window, variant) entries whose decision differs from the identity's;
          `verdict_stable`: every variant confidence lies on the identity's side of `confidence_threshold`;
          `window_starts`: the windows' first frames (those of `audio_starts_from` when given: absolute video frames).
        It reports only: nothing here enters a verdict."""
        T = self.chunk_size
        H, W = int(track_u8.shape[1]), int(track_u8.shape[2])
        names, mats = self.robustness_variants(T, H, W)
        logits = self.score_track_warps(track_u8, starts, mel_full, total_v_frames, mats, audio_starts_from=audio_starts_from)
        probs = np.array([self._calibrate(float(x)) for x in logits.cpu().flatten().tolist()], dtype=np.float64).reshape(len(starts), len(names))
        res = _agg.augmentation_stability(probs, confidence_threshold, self.confidence_smoothing, self.trim_ratio)
        res["variants"] = names
        res["window_starts"] = [int(s) for s in (audio_starts_from if audio_starts_from is not None else starts)]
        return res

    # ------------------------------------------------------------------ compression robustness (lsd_score_jpeg)
    _SAMPLING = {None: _cabi.LSD_JPEG_NONE, "444": _cabi.LSD_JPEG_444, "420": _cabi.LSD_JPEG_420}
    _CHANNEL_ORDER = {"rgb": _cabi.LSD_RGB, "bgr": _cabi.LSD_BGR}

    def _jpeg_args(self, track_u8: torch.Tensor, starts: Sequence[int], variants, channel_order: str):
        """Checks what `lsd_score_jpeg` / `lsd_jpeg_windows` would reject, as ValueError; returns (K, variants as lsd_jpeg, order)."""
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        if channel_order not in self._CHANNEL_ORDER:
            raise ValueError(f"channel_order must be 'rgb' or 'bgr', got {channel_order!r}")
        vs = [tuple(v) for v in variants]
        if not 1 <= len(vs) <= _cabi.LSD_MAX_JPEG_VARIANTS:
            raise ValueError(f"{len(vs)} JPEG variants: expected 1 to {_cabi.LSD_MAX_JPEG_VARIANTS}")
        for k, (q, sampling) in enumerate(vs):
            if sampling not in self._SAMPLING:
                raise ValueError(f"JPEG variant {k}: sampling must be '420', '444' or None, got {sampling!r}")
            if sampling is not None and not (isinstance(q, (int, np.integer)) and 1 <= int(q) <= 100):
                raise ValueError(f"JPEG variant {k}: quality must be an integer in 1..100, got {q!r}")
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        mcu = 16 if any(v[1] == "420" for v in vs) else 8
        if H % mcu or W % mcu:
            raise ValueError(f"{H}x{W} crops: JPEG sides must be multiples of {mcu} (partial MCUs are not supported)")
        T = self.chunk_size
        for i, s in enumerate(starts):
            if not 0 <= int(s) <= n_frames - T:
                raise ValueError(f"window {i} [{int(s)},{int(s) + T}) is outside the {n_frames}-frame track")
        arr = (_cabi.LsdJpeg * len(vs))(*[_cabi.LsdJpeg(int(q) if s is not None else 0, self._SAMPLING[s]) for q, s in vs])
        return len(vs), arr, self._CHANNEL_ORDER[channel_order]

    def score_track_jpeg(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int, variants,
                         chunk_a_size: int = 128, audio_starts_from: Optional[Sequence[int]] = None,
                         channel_order: str = "rgb") -> torch.Tensor:
        """`score_track_logits` with K recompressed variants per window (`lsd_score_jpeg`).  `variants`: a sequence of
        `(quality, sampling)`, sampling `"420"` (cv2's default), `"444"` or `None` (the plain window; its quality is ignored).  Every
        frame of variant k is one baseline JPEG encode + decode, bit for bit `cv2.imdecode(cv2.imencode('.jpg', frame,
        [IMWRITE_JPEG_QUALITY, quality, ...]))` on the frame in `channel_order` (`"rgb"`: converted to BGR and back around the
        round trip), built on the device.  Returns fp32 logits `(n, K)` on the device; entry (i, k) is bit for bit the logit of window
        i recompressed by variant k, with window i's audio slice."""
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        K, vc, order = self._jpeg_args(track_u8, starts, variants, channel_order)
        m = self.model
        dev = m._device()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T = self.chunk_size
        n = len(starts)
        if audio_starts_from is not None and len(audio_starts_from) != n:
            raise ValueError("audio_starts_from must have one entry per window")
        logits = torch.empty(n, K, dtype=torch.float32, device=dev)
        if n == 0:
            return logits
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n * K)
            need = L.lsd_score_jpeg_workspace_bytes(h.ptr, batch, K, T, H, W, F_, chunk_a_size, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            if n * K > batch and prec == _cabi.LSD_PREC_BF16:
                need = 2 * need      # a double workspace lets the batches overlap as in score_track_logits
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), chunk_a_size) for v in audio_starts_from])
            rc = L.lsd_score_jpeg(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, T, mel_full.data_ptr(), F_, Ta_full,
                                  int(total_v_frames), chunk_a_size, vc, K, order, prec, batch, logits.data_ptr(), ws.data_ptr(),
                                  ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return logits

    def jpeg_track_windows(self, track_u8: torch.Tensor, starts: Sequence[int], variants, channel_order: str = "rgb") -> torch.Tensor:
        """The recompressed windows `score_track_jpeg` scores, built by the same kernel (`lsd_jpeg_windows`): uint8
        `(n, K, T, H, W, 3)` on the device, window i under variant k at [i, k].  To look at what a quality does to the crop."""
        K, vc, order = self._jpeg_args(track_u8, starts, variants, channel_order)
        m = self.model
        dev = m._device()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T, n = self.chunk_size, len(starts)
        out = torch.empty((n, K, T, H, W, 3), dtype=torch.uint8, device=dev)
        if n == 0:
            return out
        track_u8 = track_u8.contiguous()
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            need = L.lsd_jpeg_windows_workspace_bytes(n, K, T, H, W)
            ws = torch.empty(max(int(need), 1), dtype=torch.uint8, device=dev)
            rc = L.lsd_jpeg_windows(h.ptr, track_u8.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*[int(s) for s in starts]), n, T, vc, K,
                                    order, out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return out

    @staticmethod
    def compression_variants() -> Tuple[List[str], List[Tuple[Optional[int], Optional[str]]]]:
        """The K = 8 recompressions of `compression_track`: names and `(quality, sampling)`.  The plain window, then 4:2:0 (cv2's
        default sampling) at qualities 95, 85, 75, 60, 45, 30 and 15."""
        qualities = (95, 85, 75, 60, 45, 30, 15)
        return ["none"] + [f"q{q}" for q in qualities], [(None, None)] + [(q, "420") for q in qualities]

    def compression_track(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                          confidence_threshold: float = 0.5, audio_starts_from: Optional[Sequence[int]] = None,
                          channel_order: str = "rgb") -> Dict[str, Any]:
        """Compression robustness of a track's verdict: one `score_track_jpeg` call with the K = 8 `compression_variants`, the
        calibrated P(real) summarised by `aggregate.augmentation_stability` (column 0, the plain window, is the identity):
          `variants`: the variant names (column order); `qualities`: their JPEG qualities (None for the plain window);
          `confidence`, `variant_confidence`, `tta_confidence`, `window_spread`, `decision_flip_rate`, `verdict_stable`: as in
          `robustness_track`;
          `lowest_stable_quality`: the lowest quality q such that every variant of quality >= q keeps the plain confidence's side
          of `confidence_threshold` (`aggregate.lowest_stable_quality`), None when the highest quality already flips it;
          `window_starts`: the windows' first frames (those of `audio_starts_from` when given: absolute video frames).
        It reports only: nothing here enters a verdict."""
        names, variants = self.compression_variants()
        logits = self.score_track_jpeg(track_u8, starts, mel_full, total_v_frames, variants, audio_starts_from=audio_starts_from,
                                       channel_order=channel_order)
        probs = np.array([self._calibrate(float(x)) for x in logits.cpu().flatten().tolist()], dtype=np.float64).reshape(len(starts), len(names))
        res = _agg.augmentation_stability(probs, confidence_threshold, self.confidence_smoothing, self.trim_ratio)
        qualities = [q for q, _ in variants]
        res["variants"] = names
        res["qualities"] = qualities
        res["lowest_stable_quality"] = _agg.lowest_stable_quality(qualities, res["variant_confidence"], res["confidence"], confidence_threshold)
        res["window_starts"] = [int(s) for s in (audio_starts_from if audio_starts_from is not None else starts)]
        return res

    # ------------------------------------------------------------------ resolution robustness (lsd_score_resizes)
    def _resize_args(self, track_u8: torch.Tensor, starts: Sequence[int], variants):
        """Checks what `lsd_score_resizes` / `lsd_resize_windows` would reject, as ValueError (all but the shared-memory limit of the
        crop size, which the library reports as ValueError before any launch); returns (K, variants as lsd_resize)."""
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        vs = [tuple(v) for v in variants]
        if not 1 <= len(vs) <= _cabi.LSD_MAX_RESIZE_VARIANTS:
            raise ValueError(f"{len(vs)} resize variants: expected 1 to {_cabi.LSD_MAX_RESIZE_VARIANTS}")
        for k, v in enumerate(vs):
            if len(v) != 2 or not all(isinstance(x, (int, np.integer)) for x in v) or not (1 <= v[0] <= H and 1 <= v[1] <= W):
                raise ValueError(f"resize variant {k}: face size must be integers (h, w) in 1..{H} x 1..{W}, got {v!r}")
        T = self.chunk_size
        for i, s in enumerate(starts):
            if not 0 <= int(s) <= n_frames - T:
                raise ValueError(f"window {i} [{int(s)},{int(s) + T}) is outside the {n_frames}-frame track")
        return len(vs), (_cabi.LsdResize * len(vs))(*[_cabi.LsdResize(int(h), int(w)) for h, w in vs])

    def score_track_resizes(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int, variants,
                            chunk_a_size: int = 128, audio_starts_from: Optional[Sequence[int]] = None) -> torch.Tensor:
        """`score_track_logits` with K face sizes per window (`lsd_score_resizes`).  `variants`: a sequence of `(h, w)`, 1 <= h <= H,
        1 <= w <= W; `(H, W)` is the plain window.  Every frame of variant k is `cv2.resize(cv2.resize(frame, (w, h), INTER_AREA),
        (W, H), INTER_LINEAR)`, bit for bit, built on the device: the crop as a face of h x w pixels in the source video would give
        it.  Returns fp32 logits `(n, K)` on the device; entry (i, k) is bit for bit the logit of window i resized by variant k, with
        window i's audio slice."""
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        K, vc = self._resize_args(track_u8, starts, variants)
        n = len(starts)
        if audio_starts_from is not None and len(audio_starts_from) != n:
            raise ValueError("audio_starts_from must have one entry per window")
        m = self.model
        dev = m._device()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T = self.chunk_size
        logits = torch.empty(n, K, dtype=torch.float32, device=dev)
        if n == 0:
            return logits
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n * K)
            need = L.lsd_score_resizes_workspace_bytes(h.ptr, batch, K, T, H, W, F_, chunk_a_size, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            if n * K > batch and prec == _cabi.LSD_PREC_BF16:
                need = 2 * need      # a double workspace lets the batches overlap as in score_track_logits
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), chunk_a_size) for v in audio_starts_from])
            rc = L.lsd_score_resizes(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, T, mel_full.data_ptr(), F_, Ta_full,
                                     int(total_v_frames), chunk_a_size, vc, K, prec, batch, logits.data_ptr(), ws.data_ptr(),
                                     ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return logits

    def resize_track_windows(self, track_u8: torch.Tensor, starts: Sequence[int], variants) -> torch.Tensor:
        """The resized windows `score_track_resizes` scores, built by the same kernel (`lsd_resize_windows`): uint8
        `(n, K, T, H, W, 3)` on the device, window i under variant k at [i, k].  To look at what a face size does to the crop."""
        K, vc = self._resize_args(track_u8, starts, variants)
        m = self.model
        dev = m._device()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T, n = self.chunk_size, len(starts)
        out = torch.empty((n, K, T, H, W, 3), dtype=torch.uint8, device=dev)
        if n == 0:
            return out
        track_u8 = track_u8.contiguous()
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            need = L.lsd_resize_windows_workspace_bytes(n, K, T, H, W)
            ws = torch.empty(max(int(need), 1), dtype=torch.uint8, device=dev)
            rc = L.lsd_resize_windows(h.ptr, track_u8.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*[int(s) for s in starts]), n, T, vc,
                                      K, out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return out

    @staticmethod
    def resolution_variants(H: int, W: int) -> Tuple[List[str], List[Tuple[int, int]]]:
        """The K = 8 face sizes of `resolution_track`: names and `(h, w)`.  The plain window, then both sides scaled by 80, 64, 56,
        48, 40, 32 and 24 over 96 and rounded (half up, at least 1): for a 96x96 crop exactly those sides, a 96 px face seen as an
        80 ... 24 px one.  With 96x96 crops the ladder takes all three INTER_AREA paths: ratio 2 (48), other integer ratios (32, 24)
        and weighted taps (the rest)."""
        sides = (80, 64, 56, 48, 40, 32, 24)
        sizes = [(int(H), int(W))] + [(max(1, (int(H) * s + 48) // 96), max(1, (int(W) * s + 48) // 96)) for s in sides]
        return ["none"] + [f"{h}x{w}" for h, w in sizes[1:]], sizes

    def resolution_track(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                         confidence_threshold: float = 0.5, audio_starts_from: Optional[Sequence[int]] = None) -> Dict[str, Any]:
        """Resolution robustness of a track's verdict: one `score_track_resizes` call with the K = 8 `resolution_variants`, the
        calibrated P(real) summarised by `aggregate.augmentation_stability` (column 0, the plain window, is the identity):
          `variants`: the variant names (column order); `sizes`: their face sizes `(h, w)` (the crop size for the plain window);
          `confidence`, `variant_confidence`, `tta_confidence`, `window_spread`, `decision_flip_rate`, `verdict_stable`: as in
          `robustness_track`;
          `lowest_stable_side`: the lowest face height h such that every variant of height >= h keeps the plain confidence's side
          of `confidence_threshold` (`aggregate.lowest_stable_quality` on the heights, the plain window left out), None when the
          largest face size already flips it;
          `window_starts`: the windows' first frames (those of `audio_starts_from` when given: absolute video frames).
        It reports only: nothing here enters a verdict."""
        H, W = int(track_u8.shape[1]), int(track_u8.shape[2])
        names, sizes = self.resolution_variants(H, W)
        logits = self.score_track_resizes(track_u8, starts, mel_full, total_v_frames, sizes, audio_starts_from=audio_starts_from)
        probs = np.array([self._calibrate(float(x)) for x in logits.cpu().flatten().tolist()], dtype=np.float64).reshape(len(starts), len(names))
        res = _agg.augmentation_stability(probs, confidence_threshold, self.confidence_smoothing, self.trim_ratio)
        heights = [None] + [h for h, _ in sizes[1:]]
        res["variants"] = names
        res["sizes"] = sizes
        res["lowest_stable_side"] = _agg.lowest_stable_quality(heights, res["variant_confidence"], res["confidence"], confidence_threshold)
        res["window_starts"] = [int(s) for s in (audio_starts_from if audio_starts_from is not None else starts)]
        return res

    # ------------------------------------------------------------------ temporal robustness (lsd_score_retimes)
    # A retime variant has one row per output frame t of the window: up to 4 taps (src, weight).  src is a frame offset from the
    # window's first track frame in -T .. 2T-1 (the library clamps the frame to the track), weights are Q15 integers >= 0 summing to
    # LSD_RETIME_ONE, and every byte is (sum w_i p_i + 16384) >> 15.  The builders below are pure, run on the CPU and return
    # (src, weight) int32 arrays of shape (T, 4); rates are exact rationals and every rounding is half up.
    @staticmethod
    def _exact_rate(x, what: str) -> Fraction:
        """`Fraction(x).limit_denominator(1001)`: 15 -> 15, 30000 / 1001 (NTSC, as a float) -> 30000/1001."""
        q = Fraction(x).limit_denominator(1001)
        if q <= 0:
            raise ValueError(f"{what} must be positive, got {x!r}")
        return q

    @staticmethod
    def _retime_table(T: int, rows) -> Tuple[np.ndarray, np.ndarray]:
        """(src, weight) int32 (T, 4) from T lists of (src, weight) taps, unused taps (0, 0); ValueError for a src outside -T .. 2T-1."""
        src = np.zeros((T, 4), np.int32)
        wt = np.zeros((T, 4), np.int32)
        for t, taps in enumerate(rows):
            for i, (s, w) in enumerate(taps):
                if not -T <= s <= 2 * T - 1:
                    raise ValueError(f"frame {t} reads frame offset {s}, outside {-T}..{2 * T - 1}: a rate or length too far out")
                src[t, i], wt[t, i] = s, w
        return src, wt

    @staticmethod
    def _capture_frame(j: int, fps: Fraction, rate: Fraction) -> int:
        """The window frame that holds capture j of a source capturing at `rate`: floor(j fps / rate + 1/2)."""
        return math.floor(j * fps / rate + Fraction(1, 2))

    @staticmethod
    def hold_retime(T: int, fps: float, rate: float) -> Tuple[np.ndarray, np.ndarray]:
        """A source that captures only at `rate` frames per second, shown at `fps`: frame t shows capture j = floor(t rate / fps),
        which sits at frame floor(j fps / rate + 1/2), never later than t.  `hold_retime(32, 15, 5)` repeats every third frame
        three times."""
        T = int(T)
        fq, rq = Predictor._exact_rate(fps, "fps"), Predictor._exact_rate(rate, "rate")
        cap = Predictor._capture_frame
        return Predictor._retime_table(T, [[(cap(math.floor(t * rq / fq), fq, rq), _cabi.LSD_RETIME_ONE)] for t in range(T)])

    @staticmethod
    def blend_retime(T: int, fps: float, rate: float) -> Tuple[np.ndarray, np.ndarray]:
        """Blended frame-rate conversion from `rate` to `fps` (ghosting): frame t is the linear blend of captures j and j + 1 at the
        fraction f = x - j, x = t rate / fps, j = floor(x); w1 = floor(f 32768 + 1/2), w0 = 32768 - w1, one tap when w1 == 0.  The
        captures sit at the frames of `hold_retime`."""
        T = int(T)
        fq, rq = Predictor._exact_rate(fps, "fps"), Predictor._exact_rate(rate, "rate")
        cap = Predictor._capture_frame
        rows = []
        for t in range(T):
            x = t * rq / fq
            j = math.floor(x)
            w1 = math.floor((x - j) * _cabi.LSD_RETIME_ONE + Fraction(1, 2))
            rows.append([(cap(j, fq, rq), _cabi.LSD_RETIME_ONE)] if w1 == 0 else
                        [(cap(j, fq, rq), _cabi.LSD_RETIME_ONE - w1), (cap(j + 1, fq, rq), w1)])
        return Predictor._retime_table(T, rows)

    @staticmethod
    def freeze_retime(T: int, at: int, length: int) -> Tuple[np.ndarray, np.ndarray]:
        """A stall that resumes live: frames at .. at + length - 1 show frame at - 1, every other frame t shows itself."""
        T, at, length = int(T), int(at), int(length)
        if at < 0 or length < 0:
            raise ValueError(f"freeze at {at} for {length} frames: both must be >= 0")
        return Predictor._retime_table(T, [[(at - 1 if at <= t < at + length else t, _cabi.LSD_RETIME_ONE)] for t in range(T)])

    @staticmethod
    def drop_retime(T: int, every: int, repeat: bool = True) -> Tuple[np.ndarray, np.ndarray]:
        """Every `every`-th source frame (s with (s + 1) % every == 0) is lost.  repeat=True: the previous frame is shown in its
        place, which keeps time.  repeat=False: the next frames are shown early, frame t shows the t-th source frame that is not
        lost, so the video drifts ahead of the audio by one frame per loss."""
        T, every = int(T), int(every)
        if every < 2:
            raise ValueError(f"drop every {every}-th frame: expected >= 2")
        if repeat:
            src: List[int] = []
            for t in range(T):
                src.append(src[-1] if (t + 1) % every == 0 else t)
        else:
            src = [s for s in range(2 * T) if (s + 1) % every != 0][:T]
        return Predictor._retime_table(T, [[(s, _cabi.LSD_RETIME_ONE)] for s in src])

    @staticmethod
    def exposure_retime(T: int, n: int) -> Tuple[np.ndarray, np.ndarray]:
        """Motion smear of an n-frame exposure, 2 <= n <= 4: frame t is the mean of frames t - c .. t - c + n - 1, c = (n - 1) // 2,
        each of weight 32768 // n, the remainder on tap c (frame t)."""
        T, n = int(T), int(n)
        if not 2 <= n <= 4:
            raise ValueError(f"exposure over {n} frames: expected 2..4")
        c, w = (n - 1) // 2, _cabi.LSD_RETIME_ONE // n
        rem = _cabi.LSD_RETIME_ONE - n * w
        return Predictor._retime_table(T, [[(t - c + i, w + (rem if i == c else 0)) for i in range(n)] for t in range(T)])

    @staticmethod
    def loss_retime(T: int, rate: float, burst: float, seed: int = 0) -> Tuple[np.ndarray, np.ndarray]:
        """Bursty frame loss (Gilbert-Elliott): a good / bad channel, P(bad -> good) = 1 / burst and P(good -> bad) =
        rate / (burst (1 - rate)), so `rate` of the frames are lost in bursts of `burst` frames on average.  Frame 0 is always
        received; frame t >= 1 draws one `np.random.default_rng(seed).random()` for its transition, and a lost frame shows the last
        received one.  Deterministic for a seed."""
        T, rate, burst = int(T), float(rate), float(burst)
        if not (0.0 <= rate < 1.0 and burst >= 1.0):
            raise ValueError(f"loss rate {rate} with bursts of {burst}: expected 0 <= rate < 1, burst >= 1")
        p_gb, p_bg = rate / (burst * (1.0 - rate)), 1.0 / burst
        if p_gb > 1.0:
            raise ValueError(f"loss rate {rate} with bursts of {burst}: P(good -> bad) = {p_gb:.3f} > 1")
        g = np.random.default_rng(int(seed))
        good, last, src = True, 0, [0]
        for t in range(1, T):
            u = g.random()
            good = (u >= p_gb) if good else (u < p_bg)
            if good:
                last = t
            src.append(last)
        return Predictor._retime_table(T, [[(s, _cabi.LSD_RETIME_ONE)] for s in src])

    @staticmethod
    def temporal_variants(T: int, fps: float = 15.0) -> Tuple[List[str], List[Tuple[np.ndarray, np.ndarray]], List[Optional[int]]]:
        """The default ladder of `temporal_track`: names, (src, weight) tables and the hold rate of each variant (None for the
        others).  The plain window (`none`); captures held from 12, 10, 8, 6 and 5 fps (`hold12` .. `hold5`) and blended from 10 fps
        (`blend10`), each only when its rate is below `fps`; stalls of 4 and 10 frames at T // 2 (`freeze4`, `freeze10`); 10 % bursty
        loss with bursts of 3 frames, seed 0 (`loss10`); every 8th frame dropped without a repeat, so the video runs ahead of the
        audio (`drift8`: 4 frames by the last frame of a 32-frame window); a 3-frame exposure (`exposure3`).  K = 12 at 15 fps."""
        T = int(T)
        P = Predictor
        fq = P._exact_rate(fps, "fps")
        names, tabs, rates = ["none"], [P._retime_table(T, [[(t, _cabi.LSD_RETIME_ONE)] for t in range(T)])], [None]
        for r in (12, 10, 8, 6, 5):
            if r < fq:
                names.append(f"hold{r}")
                tabs.append(P.hold_retime(T, fps, r))
                rates.append(r)
        if 10 < fq:
            names.append("blend10")
            tabs.append(P.blend_retime(T, fps, 10))
            rates.append(None)
        rest = [("freeze4", P.freeze_retime(T, T // 2, 4)), ("freeze10", P.freeze_retime(T, T // 2, 10)),
                ("loss10", P.loss_retime(T, 0.10, 3, 0)), ("drift8", P.drop_retime(T, 8, repeat=False)),
                ("exposure3", P.exposure_retime(T, 3))]
        for name, tab in rest:
            names.append(name)
            tabs.append(tab)
            rates.append(None)
        return names, tabs, rates

    def _retime_args(self, track_u8: torch.Tensor, starts: Sequence[int], variants):
        """Checks what `lsd_score_retimes` / `lsd_retime_windows` would reject, as ValueError; returns (K, the K*T entries as
        lsd_retime).  A variant is `(src, weight)` of shape (T, n), 1 <= n <= 4, or a bare (T,) src array: one full-weight tap."""
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        n_frames = int(track_u8.shape[0])
        T = self.chunk_size
        vs = list(variants)
        if not 1 <= len(vs) <= _cabi.LSD_MAX_RETIMES:
            raise ValueError(f"{len(vs)} retime variants: expected 1 to {_cabi.LSD_MAX_RETIMES}")
        tab = np.zeros((len(vs), T, 8), np.int32)
        for k, v in enumerate(vs):
            if isinstance(v, (tuple, list)) and len(v) == 2 and np.ndim(v[0]) == 2:
                src, wt = np.asarray(v[0]), np.asarray(v[1])
            else:
                src = np.asarray(v)
                if src.ndim != 1:
                    raise ValueError(f"retime variant {k}: expected (src, weight) of shape (T, n) or a (T,) src array, got shape {src.shape}")
                src = src[:, None]
                wt = np.full(src.shape, _cabi.LSD_RETIME_ONE, np.int64)
            if src.shape != wt.shape or src.shape[0] != T or not 1 <= src.shape[1] <= 4:
                raise ValueError(f"retime variant {k}: src {src.shape} and weight {wt.shape} must both be ({T}, n), 1 <= n <= 4")
            if src.dtype.kind not in "iu" or wt.dtype.kind not in "iu":
                raise ValueError(f"retime variant {k}: src and weight must be integers, got {src.dtype} and {wt.dtype}")
            src, wt = src.astype(np.int64), wt.astype(np.int64)
            if src.min() < -T or src.max() > 2 * T - 1:
                raise ValueError(f"retime variant {k}: src must lie in {-T}..{2 * T - 1}, got {src.min()}..{src.max()}")
            if wt.min() < 0:
                raise ValueError(f"retime variant {k}: negative weight {wt.min()}")
            bad = np.nonzero(wt.sum(axis=1) != _cabi.LSD_RETIME_ONE)[0]
            if len(bad):
                raise ValueError(f"retime variant {k}, frame {bad[0]}: weights sum to {wt[bad[0]].sum()}, not {_cabi.LSD_RETIME_ONE}")
            tab[k, :, : src.shape[1]] = src
            tab[k, :, 4: 4 + src.shape[1]] = wt
        for i, s in enumerate(starts):
            if not 0 <= int(s) <= n_frames - T:
                raise ValueError(f"window {i} [{int(s)},{int(s) + T}) is outside the {n_frames}-frame track")
        if len(starts) * len(vs) * T > 2 ** 31 - 1:
            raise ValueError(f"{len(starts)} windows x {len(vs)} retime variants: too many frames for one call")
        return len(vs), (_cabi.LsdRetime * (len(vs) * T)).from_buffer_copy(tab.tobytes())

    def score_track_retimes(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int, variants,
                            chunk_a_size: int = 128, audio_starts_from: Optional[Sequence[int]] = None) -> torch.Tensor:
        """`score_track_logits` with K retimed copies of every window (`lsd_score_retimes`).  `variants`: up to 64 retime tables,
        each `(src, weight)` of shape (T, n), 1 <= n <= 4, or a bare (T,) src array (one full-weight tap per frame), as the
        `*_retime` builders return them.  Frame t of variant k is the Q15 blend of its taps, tap frames clamp(start + src, 0,
        n_frames - 1) of the track, built on the device.  Returns fp32 logits `(n, K)` on the device; entry (i, k) is bit for bit
        the logit of window i retimed by variant k, with window i's audio slice: only the video is retimed."""
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        K, vc = self._retime_args(track_u8, starts, variants)
        n = len(starts)
        if audio_starts_from is not None and len(audio_starts_from) != n:
            raise ValueError("audio_starts_from must have one entry per window")
        m = self.model
        dev = m._device()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T = self.chunk_size
        logits = torch.empty(n, K, dtype=torch.float32, device=dev)
        if n == 0:
            return logits
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n * K)
            need = L.lsd_score_retimes_workspace_bytes(h.ptr, batch, K, T, H, W, F_, chunk_a_size, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            if n * K > batch and prec == _cabi.LSD_PREC_BF16:
                need = 2 * need      # a double workspace lets the batches overlap as in score_track_logits
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), chunk_a_size) for v in audio_starts_from])
            rc = L.lsd_score_retimes(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, T, mel_full.data_ptr(), F_, Ta_full,
                                     int(total_v_frames), chunk_a_size, vc, K, prec, batch, logits.data_ptr(), ws.data_ptr(),
                                     ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return logits

    def retime_track_windows(self, track_u8: torch.Tensor, starts: Sequence[int], variants) -> torch.Tensor:
        """The retimed windows `score_track_retimes` scores, built by the same kernel (`lsd_retime_windows`): uint8
        `(n, K, T, H, W, 3)` on the device, window i under variant k at [i, k].  To look at what a retiming does to a window."""
        K, vc = self._retime_args(track_u8, starts, variants)
        m = self.model
        dev = m._device()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        T, n = self.chunk_size, len(starts)
        out = torch.empty((n, K, T, H, W, 3), dtype=torch.uint8, device=dev)
        if n == 0:
            return out
        track_u8 = track_u8.contiguous()
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            need = L.lsd_retime_windows_workspace_bytes(n, K, T, H, W)
            ws = torch.empty(max(int(need), 1), dtype=torch.uint8, device=dev)
            rc = L.lsd_retime_windows(h.ptr, track_u8.data_ptr(), n_frames, H, W, (C.c_int32 * n)(*[int(s) for s in starts]), n, T, vc,
                                      K, out.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return out

    def temporal_track(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                       fps: float = 15.0, confidence_threshold: float = 0.5,
                       audio_starts_from: Optional[Sequence[int]] = None) -> Dict[str, Any]:
        """Temporal robustness of a track's verdict: one `score_track_retimes` call with the `temporal_variants` of the track's
        `fps`, the calibrated P(real) summarised by `aggregate.augmentation_stability` (column 0, the plain window, is the identity):
          `variants`: the variant names (column order); `rates`: the hold rate of each variant, None for the others;
          `confidence`, `variant_confidence`, `tta_confidence`, `window_spread`, `decision_flip_rate`, `verdict_stable`: as in
          `robustness_track`;
          `lowest_stable_fps`: the lowest hold rate r such that every hold variant of rate >= r keeps the plain confidence's side of
          `confidence_threshold` (`aggregate.lowest_stable_quality` on `rates`), None when the highest rate already flips it or no
          rate is below `fps`;
          `window_starts`: the windows' first frames (those of `audio_starts_from` when given: absolute video frames).
        Frames just outside a window are read from the track, so give the whole track.  It reports only: nothing here enters a
        verdict."""
        names, tabs, rates = self.temporal_variants(self.chunk_size, fps)
        logits = self.score_track_retimes(track_u8, starts, mel_full, total_v_frames, tabs, audio_starts_from=audio_starts_from)
        return self._temporal_report(logits.cpu().numpy(), names, rates, confidence_threshold,
                                     audio_starts_from if audio_starts_from is not None else starts)

    def _temporal_report(self, logits: np.ndarray, names: List[str], rates: List[Optional[int]], confidence_threshold: float,
                         window_starts: Sequence[int]) -> Dict[str, Any]:
        """`temporal_track`'s dict from (n, K) logits of the `temporal_variants` columns `names` / `rates`."""
        probs = np.array([self._calibrate(float(x)) for x in np.asarray(logits).flatten().tolist()],
                         dtype=np.float64).reshape(len(window_starts), len(names))
        res = _agg.augmentation_stability(probs, confidence_threshold, self.confidence_smoothing, self.trim_ratio)
        res["variants"] = names
        res["rates"] = rates
        res["lowest_stable_fps"] = _agg.lowest_stable_quality(rates, res["variant_confidence"], res["confidence"], confidence_threshold)
        res["window_starts"] = [int(s) for s in window_starts]
        return res

    # ------------------------------------------------------------------ audio robustness (lsd_degrade_audio, lsd_score_audio_clips)
    _AD_KEYS = (("rt60", _cabi.LSD_AD_REVERB, 0.05, 2.0), ("snr_db", _cabi.LSD_AD_NOISE, -20.0, 60.0),
                ("gain_db", _cabi.LSD_AD_CLIP, 0.0, 40.0))

    @classmethod
    def _degradation(cls, k: int, v) -> "_cabi.LsdAudioDegradation":
        """One variant as lsd_audio_degradation, checked as lsd_degrade_audio checks it (ValueError).  A dict enables the stages whose
        keys it has: `rt60`, `snr_db`, `gain_db`, `band_rate`, `mulaw` (True); `seed` (default 0) keys the generator.  A tuple is
        `(stages, rt60, snr_db, gain_db, band_rate, seed)` with the LSD_AD_* bits."""
        if isinstance(v, dict):
            unknown = set(v) - {"rt60", "snr_db", "gain_db", "band_rate", "mulaw", "seed"}
            if unknown:
                raise ValueError(f"audio degradation {k}: unknown keys {sorted(unknown)}")
            stages = sum(bit for key, bit, _, _ in cls._AD_KEYS if key in v)
            stages |= _cabi.LSD_AD_BAND if "band_rate" in v else 0
            stages |= _cabi.LSD_AD_MULAW if v.get("mulaw", False) else 0
            t = (stages, v.get("rt60", 0.0), v.get("snr_db", 0.0), v.get("gain_db", 0.0), v.get("band_rate", 0), v.get("seed", 0))
        else:
            t = tuple(v)
            if len(t) != 6:
                raise ValueError(f"audio degradation {k}: expected (stages, rt60, snr_db, gain_db, band_rate, seed), got {v!r}")
        stages, rt60, snr, gain, rate, seed = t
        all_bits = _cabi.LSD_AD_REVERB | _cabi.LSD_AD_NOISE | _cabi.LSD_AD_CLIP | _cabi.LSD_AD_BAND | _cabi.LSD_AD_MULAW
        if not isinstance(stages, (int, np.integer)) or int(stages) & ~all_bits or int(stages) < 0:
            raise ValueError(f"audio degradation {k}: bad stage bits {stages!r}")
        stages = int(stages)
        for (key, bit, lo, hi), val in zip(cls._AD_KEYS, (rt60, snr, gain)):
            if stages & bit and not (np.isfinite(float(val)) and lo <= float(np.float32(val)) <= hi):
                raise ValueError(f"audio degradation {k}: {key} {val!r} is outside [{lo:g}, {hi:g}]")
        if stages & _cabi.LSD_AD_BAND and rate not in (8000, 4000):
            raise ValueError(f"audio degradation {k}: band_rate must be 8000 or 4000, got {rate!r}")
        if not (isinstance(seed, (int, np.integer)) and 0 <= int(seed) < 2 ** 32):
            raise ValueError(f"audio degradation {k}: seed must be an integer in [0, 2^32), got {seed!r}")
        return _cabi.LsdAudioDegradation(stages, float(rt60), float(snr), float(gain), int(rate) if stages & _cabi.LSD_AD_BAND else 0,
                                         int(seed))

    def degrade_audio(self, pcm, variants) -> torch.Tensor:
        """K degraded copies of one 16 kHz mono clip (`lsd_degrade_audio`): fp32 `(K, n)` on the device, variant k at row k.  `pcm`: a
        1-D float tensor or array.  `variants`: dicts or `lsd_audio_degradation`-shaped tuples (`_degradation`); the stages run in the
        order reverb, noise, clip, band, mu-law, and a variant with none copies the clip."""
        vs = [self._degradation(k, v) for k, v in enumerate(variants)]
        K = len(vs)
        if not 1 <= K <= _cabi.LSD_MAX_AUDIO_DEGRADATIONS:
            raise ValueError(f"{K} audio degradations: expected 1 to {_cabi.LSD_MAX_AUDIO_DEGRADATIONS}")
        x = (pcm if isinstance(pcm, torch.Tensor) else torch.from_numpy(np.asarray(pcm)))
        if x.dim() != 1 or x.numel() < 1:
            raise ValueError(f"pcm must be a non-empty 1-D clip, got shape {tuple(x.shape)}")
        m = self.model
        dev = m._device()
        x = x.to(device=dev, dtype=torch.float32).contiguous()
        n = int(x.numel())
        out = torch.empty((K, n), dtype=torch.float32, device=dev)
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            ws = torch.empty(int(L.lsd_degrade_audio_workspace_bytes(n, K)), dtype=torch.uint8, device=dev)
            rc = L.lsd_degrade_audio(h.ptr, x.data_ptr(), n, (_cabi.LsdAudioDegradation * K)(*vs), K, out.data_ptr(), ws.data_ptr(),
                                     ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return out

    def score_track_audio_clips(self, track_u8: torch.Tensor, starts: Sequence[int], mels: torch.Tensor, total_v_frames: int,
                                chunk_a_size: int = 128, audio_starts_from: Optional[Sequence[int]] = None) -> torch.Tensor:
        """`score_track_logits` against K clip log-mels at once (`lsd_score_audio_clips`).  `mels`: `(K, F, T_full)` on the device,
        e.g. the log-mels of `degrade_audio`'s clips, or of the clip run through a lossy codec on the host.  The video side of a window
        runs once for all K.  Returns fp32 logits `(n, K)` on the device; column k is bit for bit `score_track_logits(track, starts,
        mels[k:k+1], ...)`."""
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        if mels.dim() != 3 or mels.shape[2] < 1:
            raise ValueError(f"mels must be (K, F, T_full), got {tuple(mels.shape)}")
        K = int(mels.shape[0])
        if not 1 <= K <= _cabi.LSD_MAX_AUDIO_DEGRADATIONS:
            raise ValueError(f"{K} clips: expected 1 to {_cabi.LSD_MAX_AUDIO_DEGRADATIONS}")
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        F_, Ta_full = int(mels.shape[1]), int(mels.shape[2])
        T, Ta = self.chunk_size, int(chunk_a_size)
        n = len(starts)
        if audio_starts_from is not None and len(audio_starts_from) != n:
            raise ValueError("audio_starts_from must have one entry per window")
        for i, s in enumerate(starts):
            if not 0 <= int(s) <= n_frames - T:
                raise ValueError(f"window {i} [{int(s)},{int(s) + T}) is outside the {n_frames}-frame track")
        m = self.model
        dev = m._device()
        logits = torch.empty(n, K, dtype=torch.float32, device=dev)
        if n == 0:
            return logits
        track_u8 = track_u8.contiguous()
        mels = mels.to(torch.float32).contiguous()
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            prec = m._precision()
            batch = min(self.batch_size, n)
            need = L.lsd_score_audio_clips_workspace_bytes(h.ptr, batch, K, T, H, W, F_, Ta, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            ws = m._workspace(need, dev)
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), Ta) for v in audio_starts_from])
            rc = L.lsd_score_audio_clips(h.ptr, track_u8.data_ptr(), n_frames, H, W, st, ast, n, T, mels.data_ptr(), F_, Ta_full,
                                         int(total_v_frames), Ta, K, prec, batch, logits.data_ptr(), ws.data_ptr(), ws.numel(),
                                         torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return logits

    @staticmethod
    def audio_degradation_variants() -> Tuple[List[str], List[Dict[str, Any]]]:
        """The K = 10 degradations of `audio_robustness_track`: names and variant dicts.  The clean clip, white noise at 30, 20, 10, 5
        and 0 dB SNR, a phone line (8 kHz band + mu-law), a phone line in a noisy room (10 dB, then the phone line), a reverberant
        room (rt60 0.5 s) and a microphone overdriven by 12 dB."""
        ladder = (30, 20, 10, 5, 0)
        names = ["none"] + [f"snr{s}" for s in ladder] + ["phone", "noisy_phone", "reverb", "clipped"]
        variants = [{}] + [{"snr_db": float(s)} for s in ladder] + [
            {"band_rate": 8000, "mulaw": True}, {"snr_db": 10.0, "band_rate": 8000, "mulaw": True}, {"rt60": 0.5}, {"gain_db": 12.0}]
        return names, variants

    def audio_robustness_track(self, track_u8: torch.Tensor, starts: Sequence[int], pcm, total_v_frames: int,
                               confidence_threshold: float = 0.5, variants=None,
                               audio_starts_from: Optional[Sequence[int]] = None) -> Dict[str, Any]:
        """Audio robustness of a track's verdict: `degrade_audio` on the clip's PCM, the log-mel of the K copies in one call
        (`audio.logmel_db`), one `score_track_audio_clips` call, and the calibrated P(real) summarised by
        `aggregate.augmentation_stability` (column 0 is the identity).  `variants`: `(names, variants)` as `audio_degradation_variants`
        returns them (the default), column 0 the clean clip.  Returns:
          `variants`: the variant names (column order); `snr_db`: the SNR of the variants on the noise ladder (noise only), None for
          the others;
          `confidence`, `variant_confidence`, `tta_confidence`, `window_spread`, `decision_flip_rate`, `verdict_stable`: as in
          `robustness_track`;
          `lowest_stable_snr`: `aggregate.lowest_stable_quality` on the SNR ladder (a higher SNR is milder noise, the ordering of JPEG
          quality): the lowest SNR down to which every noise variant keeps the clean confidence's side of `confidence_threshold`,
          None when the mildest already flips it;
          `window_starts`: the windows' first frames (those of `audio_starts_from` when given: absolute video frames).
        It reports only: nothing here enters a verdict."""
        from .audio import logmel_db
        names, vs = variants if variants is not None else self.audio_degradation_variants()
        names = list(names)
        if len(names) != len(vs):
            raise ValueError(f"{len(names)} names for {len(vs)} audio degradations")
        clips = self.degrade_audio(pcm, vs)
        mels = logmel_db(clips)
        logits = self.score_track_audio_clips(track_u8, starts, mels, total_v_frames, audio_starts_from=audio_starts_from)
        probs = np.array([self._calibrate(float(x)) for x in logits.cpu().flatten().tolist()], dtype=np.float64).reshape(len(starts), len(names))
        res = _agg.augmentation_stability(probs, confidence_threshold, self.confidence_smoothing, self.trim_ratio)
        degr = [self._degradation(k, v) for k, v in enumerate(vs)]
        snr = [float(d.snr_db) if d.stages == _cabi.LSD_AD_NOISE else None for d in degr]
        res["variants"] = names
        res["snr_db"] = snr
        res["lowest_stable_snr"] = _agg.lowest_stable_quality(snr, res["variant_confidence"], res["confidence"], confidence_threshold)
        res["window_starts"] = [int(s) for s in (audio_starts_from if audio_starts_from is not None else starts)]
        return res

    def score_track(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int):
        logits = self.score_track_logits(track_u8, starts, mel_full, total_v_frames)
        confs = [self._calibrate(float(x)) for x in logits.cpu().tolist()]
        return self._robust_confidence(confs), confs

    # ------------------------------------------------------------------ speaking alignment / mouth motion (SURVEY.md §8f-2)
    def window_speech_stats(self, track_u8: torch.Tensor, starts: Sequence[int], mel_full: torch.Tensor, total_v_frames: int,
                            chunk_a_size: int = 128, audio_starts_from: Optional[Sequence[int]] = None):
        """Per-window `(speaking_alignment, mouth_motion_energy, audio_energy)` fp32 device tensors for the windows of a
        uint8 track: the statistics `_predict_long_video` computes per window with `_speaking_alignment_score`
        (predictor.py:333-370) and `_mouth_motion_energy_check` (:374-419).  Frame-difference energies are computed once
        per frame pair of the track (`lsd_track_motion`), then combined per window (`lsd_speech_stats`)."""
        m = self.model
        dev = m._device()
        if track_u8.dtype != torch.uint8 or track_u8.dim() != 4 or track_u8.shape[3] != 3:
            raise ValueError(f"track must be uint8 (n_frames, H, W, 3), got {track_u8.dtype} {tuple(track_u8.shape)}")
        if mel_full.dim() != 3 or mel_full.shape[0] != 1:
            raise ValueError(f"mel_full must be (1, F, T_full), got {tuple(mel_full.shape)}")
        n = len(starts)
        out = [torch.empty(n, dtype=torch.float32, device=dev) for _ in range(3)]
        if n == 0:
            return tuple(out)
        track_u8 = track_u8.contiguous()
        mel_full = mel_full.to(torch.float32).contiguous()
        n_frames, H, W = int(track_u8.shape[0]), int(track_u8.shape[1]), int(track_u8.shape[2])
        F_, Ta_full = int(mel_full.shape[1]), int(mel_full.shape[2])
        motion = torch.zeros(2, max(1, n_frames - 1), dtype=torch.float32, device=dev)
        idx = torch.empty(2 * n, dtype=torch.int32, device=dev)
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            stream = torch.cuda.current_stream(dev).cuda_stream
            _cabi.check(h.ptr, L.lsd_track_motion(h.ptr, track_u8.data_ptr(), _cabi.LSD_U8, _cabi.LSD_NDHWC, n_frames, H, W,
                                                  motion[0].data_ptr(), motion[1].data_ptr(), stream))
            st = (C.c_int32 * n)(*[int(s) for s in starts])
            ast = None
            if audio_starts_from is not None:
                ast = (C.c_int32 * n)(*[self._audio_start(int(v), Ta_full, int(total_v_frames), chunk_a_size) for v in audio_starts_from])
            rc = L.lsd_speech_stats(h.ptr, motion[0].data_ptr(), motion[1].data_ptr(), n_frames, st, ast, n, self.chunk_size,
                                    mel_full.data_ptr(), F_, Ta_full, int(total_v_frames), chunk_a_size, out[0].data_ptr(),
                                    out[1].data_ptr(), out[2].data_ptr(), idx.data_ptr(), stream)
            _cabi.check(h.ptr, rc)
        return tuple(out)

    def _speaking_alignment_score(self, visual_np: np.ndarray, audio_np: np.ndarray) -> float:
        """Same contract as the reference static method (predictor.py:333-370): `(3,T,H,W)` float32 crop in [0,1] +
        `(1,F,T_a)` log-mel -> score in [0,1]; computed on the device."""
        m = self.model
        dev = m._device()
        v = torch.from_numpy(np.ascontiguousarray(visual_np, dtype=np.float32)).to(dev)
        a = torch.from_numpy(np.ascontiguousarray(audio_np, dtype=np.float32)).to(dev)
        T, H, W = int(v.shape[1]), int(v.shape[2]), int(v.shape[3])
        Ta = int(a.shape[2])
        if T < 2 or Ta < 2:
            return 0.5
        motion = torch.zeros(2, T - 1, dtype=torch.float32, device=dev)
        out = torch.empty(3, dtype=torch.float32, device=dev)
        idx = torch.empty(2, dtype=torch.int32, device=dev)
        with m._lsd_lock:
            h = m._ensure_handle(dev)
            L = _cabi.lib()
            stream = torch.cuda.current_stream(dev).cuda_stream
            _cabi.check(h.ptr, L.lsd_track_motion(h.ptr, v.data_ptr(), _cabi.LSD_F32, _cabi.LSD_NCDHW, T, H, W,
                                                  motion[0].data_ptr(), motion[1].data_ptr(), stream))
            st = (C.c_int32 * 1)(0)
            rc = L.lsd_speech_stats(h.ptr, motion[0].data_ptr(), motion[1].data_ptr(), T, st, st, 1, T, a.data_ptr(), int(a.shape[1]), Ta,
                                    T, Ta, out[0:1].data_ptr(), out[1:2].data_ptr(), out[2:3].data_ptr(), idx.data_ptr(), stream)
            _cabi.check(h.ptr, rc)
        return float(out[0].item())

    def mouth_motion_checks(self, mouth_motion: Sequence[float], audio_energy: Sequence[float], mouth_motion_low_threshold: float = 0.015,
                            audio_energy_high_threshold: float = -25.0, audio_energy_low_threshold: float = -50.0) -> List[dict]:
        """Decision logic of `_mouth_motion_energy_check` (predictor.py:403-419) on the per-window statistics."""
        res = []
        for motion, energy in zip(mouth_motion, audio_energy):
            motion, energy = float(motion), float(energy)
            if energy > audio_energy_high_threshold and motion < mouth_motion_low_threshold:
                r = "likely_fake"
            elif energy < audio_energy_low_threshold and motion < mouth_motion_low_threshold:
                r = "uncertain"
            else:
                r = "no_issue"
            res.append({"audio_energy": round(energy, 4), "mouth_motion_energy": round(motion, 6), "check_result": r})
        return res

    @staticmethod
    def aggregate_mouth_motion_checks(checks: Sequence[dict], max_samples: int = 5) -> dict:
        """`_aggregate_mouth_motion_check` (predictor.py:463-523): sample up to `max_samples` evenly spaced windows (always the
        last one), majority vote with the conservative `uncertain` rule."""
        n = len(checks)
        if n == 0:
            return {"check_result": "no_data", "audio_energy": 0.0, "mouth_motion_energy": 0.0, "samples_checked": 0}
        if n <= max_samples:
            indices = list(range(n))
        else:
            step = n / max_samples
            indices = [int(i * step) for i in range(max_samples)]
            if (n - 1) not in indices:
                indices[-1] = n - 1
        counts = {"likely_fake": 0, "uncertain": 0, "no_issue": 0}
        energies, motions = [], []
        for i in indices:
            c = checks[i]
            counts[c["check_result"]] = counts.get(c["check_result"], 0) + 1
            energies.append(float(c["audio_energy"]))
            motions.append(float(c["mouth_motion_energy"]))
        k = len(indices)
        if counts["uncertain"] > k // 2:
            agg = "uncertain"
        elif counts["likely_fake"] > counts["uncertain"] + counts["no_issue"]:
            agg = "likely_fake"
        else:
            agg = "no_issue"
        return {"check_result": agg, "audio_energy": round(float(np.median(energies)), 4),
                "mouth_motion_energy": round(float(np.median(motions)), 6), "samples_checked": k, "counts": counts}

    # ------------------------------------------------------------------ decision (predictor.py:856-1155, :1235)
    def aggregate_long_video(self, window_confs, window_speaking, window_vad_weights=None, mouth_check_result: str = "no_data", **gates):
        """Final `real` / `fake` / `uncertain` decision from per-window confidences; see `lipsync_b200.aggregate`."""
        from .aggregate import aggregate_long_video
        return aggregate_long_video(window_confs, window_speaking, window_vad_weights, mouth_check_result,
                                    confidence_smoothing=self.confidence_smoothing, trim_ratio=self.trim_ratio, **gates)

    # ------------------------------------------------------------------ multi-GPU (SURVEY.md §8e)
    def score_windows_sharded(self, n_windows: int, score_range: Callable[[int, int], torch.Tensor],
                              world_size: int, rank: int) -> torch.Tensor:
        """Each rank scores its contiguous block `[lo,hi)` with `score_range(lo, hi) -> logits`, then one
        all-gather returns all `n_windows` fp32 logits on every rank (rank 0 runs the host aggregation)."""
        lo, hi = partition_windows(n_windows, world_size, rank)
        local = score_range(lo, hi) if hi > lo else torch.empty(0, dtype=torch.float32, device=self.device)
        return gather_logits(local, n_windows, world_size, rank)
