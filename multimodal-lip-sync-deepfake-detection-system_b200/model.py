"""`LipSyncModel`: host-side mirror of the reference module boundary (app/models/lip_sync_model.py:14-145).

Same constructor defaults, `forward(visual, audio, return_aux=False) -> logits (B,)`, `predict`, and a
`state_dict()` / `load_state_dict(strict=True)` with the reference's 270 keys, so `Predictor` code such as
    model = LipSyncModel(); model.load_state_dict(state, strict=True); model.half(); model.to(device); model.eval()
(app/inference/predictor.py:139,187-200) runs unchanged.  The module holds the parameters only as the
weight boundary; every numeric op of `forward` runs in `liblsd_b200.so` through its C-ABI.
"""
from __future__ import annotations

import ctypes as C
import math
import threading
from typing import Dict, Optional, Tuple, Union

import torch
from torch import Tensor, nn

from . import _cabi
from .state_spec import BUFFER_SUFFIXES, state_spec

_DTYPES = {torch.float32: _cabi.LSD_F32, torch.float16: _cabi.LSD_F16, torch.bfloat16: _cabi.LSD_BF16, torch.uint8: _cabi.LSD_U8}


class _Node(nn.Module):
    """Anonymous container used to rebuild the reference's dotted parameter names."""


def _init_tensor(name: str, shape) -> Tensor:
    # Initialisation family of the reference (visual_encoder.py:158-164, audio_encoder.py:162-171,
    # temporal.py:31-32, artifact_detector.py:14-21); real use always loads a checkpoint.
    if name.endswith("num_batches_tracked"):
        return torch.tensor(0, dtype=torch.int64)
    if name.endswith("running_mean"):
        return torch.zeros(shape)
    if name.endswith("running_var"):
        return torch.ones(shape)
    if name.endswith("laplacian.weight"):
        k = torch.tensor([[0.0, 1.0, 0.0], [1.0, -4.0, 1.0], [0.0, 1.0, 0.0]])
        w = torch.zeros(shape)
        for i in range(3):
            w[i, i] = k
        return w
    if name == "temporal.cls_token":
        return torch.randn(shape) * 0.02
    if len(shape) >= 3:
        fan_out = shape[0] * math.prod(shape[2:])
        return torch.randn(shape) * math.sqrt(2.0 / fan_out)
    if len(shape) == 2:
        bound = 1.0 / math.sqrt(shape[1])
        return (torch.rand(shape) * 2 - 1) * bound
    if name.endswith(".weight"):
        return torch.ones(shape)
    return torch.zeros(shape)


class LipSyncModel(nn.Module):
    """Drop-in for the reference `LipSyncModel` on the window-scoring path (inference only)."""

    def __init__(
        self,
        visual_feature_dim: int = 256,
        audio_feature_dim: int = 256,
        embed_dim: int = 256,
        detect_artifacts: bool = True,
        cross_modal_heads: int = 8,
        temporal_layers: int = 4,
        temporal_heads: int = 8,
        temporal_pre_conv: bool = True,
        use_delta_artifact: bool = True,
        use_high_freq_artifact: bool = True,
        preserve_audio_temporal: bool = True,
    ) -> None:
        super().__init__()
        cfg = (visual_feature_dim, audio_feature_dim, embed_dim, detect_artifacts, cross_modal_heads, temporal_layers,
               temporal_heads, temporal_pre_conv, use_delta_artifact, use_high_freq_artifact, preserve_audio_temporal)
        if cfg != (256, 256, 256, True, 8, 4, 8, True, True, True, True):
            raise NotImplementedError(
                "lipsync_b200.LipSyncModel implements the default R2Plus1D-Sync configuration only (the one every "
                "reference caller constructs: predictor.py:139, train.py, validate_pipeline.py)")
        self.detect_artifacts = True
        for name, shape in state_spec().items():
            self._register(name, _init_tensor(name, tuple(shape)))
        self.eval()
        self._lsd_lock = threading.RLock()
        self._lsd_handle: Optional[_cabi.Handle] = None
        self._lsd_dirty = True
        self._lsd_ws: Optional[Tensor] = None
        self._lsd_plan_dtype = None
        #: "auto": fp32 parameters -> fp32 CUDA-core path, half/bfloat16 parameters -> bf16 tcgen05 path.
        self.compute_precision = "auto"

    # ------------------------------------------------------------------ parameter tree
    def _register(self, name: str, value: Tensor) -> None:
        parts = name.split(".")
        mod: nn.Module = self
        for p in parts[:-1]:
            if p not in mod._modules:
                mod.add_module(p, _Node())
            mod = mod._modules[p]
        if name.endswith(BUFFER_SUFFIXES):
            mod.register_buffer(parts[-1], value)
        else:
            mod.register_parameter(parts[-1], nn.Parameter(value, requires_grad=False))

    def _apply(self, fn, *args, **kwargs):  # .to() / .half() / .float() / .cuda()
        self._lsd_dirty = True
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        self._lsd_dirty = True
        return super().load_state_dict(state_dict, strict=strict, assign=assign)

    def refresh_weights(self) -> None:
        """Call after editing parameters in place; the packed device copy is rebuilt on the next forward."""
        self._lsd_dirty = True

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("lipsync_b200.LipSyncModel is inference-only (the backward pass is out of scope)")
        return super().train(False)

    # ------------------------------------------------------------------ C-ABI plumbing
    def _device(self) -> torch.device:
        return self.classifier.net._modules["4"].weight.device

    def _dtype(self) -> torch.dtype:
        return self.classifier.net._modules["4"].weight.dtype

    def _precision(self) -> int:
        if self.compute_precision == "fp32":
            return _cabi.LSD_PREC_FP32
        if self.compute_precision == "bf16":
            return _cabi.LSD_PREC_BF16
        return _cabi.LSD_PREC_FP32 if self._dtype() == torch.float32 else _cabi.LSD_PREC_BF16

    def _ensure_handle(self, device: torch.device) -> _cabi.Handle:
        if device.type != "cuda":
            raise RuntimeError(
                "lipsync_b200.LipSyncModel runs only on an sm_100 CUDA device (call .to('cuda')); there is no CPU fallback")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        if self._lsd_handle is None or self._lsd_handle.device_index != idx:
            if self._lsd_handle is not None:
                self._lsd_handle.close()
            self._lsd_handle = _cabi.Handle(idx)
            self._lsd_dirty = True
        if self._lsd_dirty:
            sd = self.state_dict()
            keep = []
            arr = (_cabi.LsdTensor * len(sd))()
            for i, (k, v) in enumerate(sd.items()):
                is_i64 = v.dtype == torch.int64
                t = v.detach().to("cpu", torch.int64 if is_i64 else torch.float32).contiguous()
                keep.append(t)
                arr[i].name = k.encode()
                arr[i].dtype = _cabi.LSD_I64 if is_i64 else _cabi.LSD_F32
                arr[i].ndim = t.dim()
                for d, s in enumerate(t.shape):
                    arr[i].shape[d] = s
                arr[i].data = t.data_ptr()
            _cabi.check(self._lsd_handle.ptr, _cabi.lib().lsd_load_weights(self._lsd_handle.ptr, arr, len(sd)))
            self._lsd_dirty = False
        return self._lsd_handle

    def _workspace(self, nbytes: int, device: torch.device) -> Tensor:
        if self._lsd_ws is None or self._lsd_ws.device != device or self._lsd_ws.numel() < nbytes:
            self._lsd_ws = None
            self._lsd_ws = torch.empty(int(nbytes * 1.05) + 1024, dtype=torch.uint8, device=device)
            # a fresh allocation may reuse the address of the freed one: the library must not trust remembered padding
            if self._lsd_handle is not None:
                _cabi.lib().lsd_workspace_invalidate(self._lsd_handle.ptr)
        return self._lsd_ws

    # ------------------------------------------------------------------ forward
    def forward(self, visual: Tensor, audio: Tensor, return_aux: bool = False,
                video_layout: str = "NCDHW") -> Union[Tensor, Tuple[Tensor, Dict[str, Tensor]]]:
        """visual `(B,3,T,H,W)` (or `(B,T,H,W,3)` with `video_layout="NDHWC"`; uint8 is scaled by 1/255),
        audio `(B,1,F,T_a)` log-mel dB.  Returns logits `(B,)` for P(REAL) (lip_sync_model.py:86-136)."""
        if visual.dim() != 5:
            raise ValueError(f"VisualEncoder expected input of shape (B, 3, T, H, W), got {tuple(visual.shape)}")
        if audio.dim() != 4:
            raise ValueError(f"AudioEncoder expected input of shape (B, 1, F, T), got {tuple(audio.shape)}")
        if video_layout == "NCDHW":
            B, Cv, T, H, W = visual.shape
            layout = _cabi.LSD_NCDHW
        elif video_layout == "NDHWC":
            B, T, H, W, Cv = visual.shape
            layout = _cabi.LSD_NDHWC
        else:
            raise ValueError(f"unknown video_layout {video_layout!r}")
        if Cv != 3:
            raise ValueError(f"VisualEncoder expected 3 input channels, got {Cv}")
        if audio.shape[0] != B or audio.shape[1] != 1:
            raise ValueError(f"AudioEncoder expected input of shape ({B}, 1, F, T), got {tuple(audio.shape)}")
        if visual.dtype not in _DTYPES or audio.dtype not in _DTYPES or audio.dtype == torch.uint8:
            raise RuntimeError(f"unsupported input dtypes {visual.dtype}/{audio.dtype}")
        dev = self._device()
        if visual.device != dev or audio.device != dev:
            raise RuntimeError(f"inputs must live on the module's device {dev} (got {visual.device}, {audio.device})")
        F_, Ta = int(audio.shape[2]), int(audio.shape[3])
        out_dtype = visual.dtype if visual.dtype.is_floating_point else torch.float32
        with self._lsd_lock:  # forward may be entered from two threads (api/routes.py:45 + worker/worker.py:53)
            h = self._ensure_handle(dev)
            L = _cabi.lib()
            prec = self._precision()
            visual = visual.contiguous()
            audio = audio.contiguous()
            logits = torch.empty(int(B), dtype=torch.float32, device=dev)
            if B == 0:
                return (logits.to(out_dtype), {}) if return_aux else logits.to(out_dtype)
            need = L.lsd_workspace_bytes(h.ptr, int(B), int(T), int(H), int(W), F_, Ta, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            ws = self._workspace(need, dev)
            aux_t = None
            aux_p = None
            if return_aux:
                ta_tok = L.lsd_audio_tokens(Ta)
                aux_t = {
                    "visual_tokens": torch.empty(B, T, 256, dtype=torch.float32, device=dev),
                    "audio_tokens": torch.empty(B, ta_tok, 256, dtype=torch.float32, device=dev),
                    "fused_tokens": torch.empty(B, T, 256, dtype=torch.float32, device=dev),
                    "cls_output": torch.empty(B, 256, dtype=torch.float32, device=dev),
                }
                aux_s = _cabi.LsdAux(aux_t["visual_tokens"].data_ptr(), aux_t["audio_tokens"].data_ptr(),
                                     aux_t["fused_tokens"].data_ptr(), aux_t["cls_output"].data_ptr())
                aux_p = C.byref(aux_s)
            stream = torch.cuda.current_stream(dev).cuda_stream
            rc = L.lsd_forward(h.ptr, visual.data_ptr(), _DTYPES[visual.dtype], layout, audio.data_ptr(), _DTYPES[audio.dtype],
                               int(B), int(T), int(H), int(W), F_, Ta, prec, logits.data_ptr(), aux_p,
                               ws.data_ptr(), ws.numel(), stream)
            _cabi.check(h.ptr, rc)
            self._lsd_plan_dtype = prec
        logits = logits.to(out_dtype)
        if not return_aux:
            return logits
        return logits, {k: v.to(out_dtype) for k, v in aux_t.items()}

    def forward_audio_variants(self, visual: Tensor, audio: Tensor) -> Tensor:
        """Score K audio windows against every video: visual `(B,3,T,H,W)`, audio `(B,K,1,F,T_a)` -> logits `(B,K)`.
        `[:, k]` is bit for bit `forward(visual, audio[:, k])`; the visual encoder and the artifact branch run once per video
        (`lsd_forward_audio_variants`).  1 <= K <= 64."""
        if visual.dim() != 5:
            raise ValueError(f"VisualEncoder expected input of shape (B, 3, T, H, W), got {tuple(visual.shape)}")
        if audio.dim() != 5:
            raise ValueError(f"expected audio variants of shape (B, K, 1, F, T), got {tuple(audio.shape)}")
        B, Cv, T, H, W = visual.shape
        K = int(audio.shape[1])
        if Cv != 3:
            raise ValueError(f"VisualEncoder expected 3 input channels, got {Cv}")
        if audio.shape[0] != B or audio.shape[2] != 1:
            raise ValueError(f"expected audio variants of shape ({B}, K, 1, F, T), got {tuple(audio.shape)}")
        if not 1 <= K <= _cabi.LSD_MAX_AUDIO_VARIANTS:
            raise ValueError(f"K = {K} audio variants: expected 1 <= K <= {_cabi.LSD_MAX_AUDIO_VARIANTS}")
        if visual.dtype not in _DTYPES or audio.dtype not in _DTYPES or audio.dtype == torch.uint8:
            raise RuntimeError(f"unsupported input dtypes {visual.dtype}/{audio.dtype}")
        dev = self._device()
        if visual.device != dev or audio.device != dev:
            raise RuntimeError(f"inputs must live on the module's device {dev} (got {visual.device}, {audio.device})")
        F_, Ta = int(audio.shape[3]), int(audio.shape[4])
        out_dtype = visual.dtype if visual.dtype.is_floating_point else torch.float32
        logits = torch.empty(int(B), K, dtype=torch.float32, device=dev)
        if B == 0:
            return logits.to(out_dtype)
        with self._lsd_lock:
            h = self._ensure_handle(dev)
            L = _cabi.lib()
            prec = self._precision()
            visual = visual.contiguous()
            audio = audio.contiguous()
            need = L.lsd_forward_audio_variants_workspace_bytes(h.ptr, int(B), K, int(T), int(H), int(W), F_, Ta, prec)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            ws = self._workspace(need, dev)
            rc = L.lsd_forward_audio_variants(h.ptr, visual.data_ptr(), _DTYPES[visual.dtype], _cabi.LSD_NCDHW, audio.data_ptr(),
                                              _DTYPES[audio.dtype], int(B), K, int(T), int(H), int(W), F_, Ta, prec, logits.data_ptr(),
                                              ws.data_ptr(), ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
            self._lsd_plan_dtype = prec
        return logits.to(out_dtype)

    def forward_into(self, visual: Tensor, audio: Tensor, logits: Tensor, workspace: Tensor) -> None:
        """Allocation-free forward for CUDA-graph capture: device `visual (B,3,T,H,W)` / `audio (B,1,F,T_a)` (contiguous),
        fp32 device `logits (B,)`, caller-owned `workspace` (uint8, >= `workspace_bytes(...)`), current stream."""
        B, _, T, H, W = visual.shape
        F_, Ta = int(audio.shape[2]), int(audio.shape[3])
        dev = self._device()
        with self._lsd_lock:
            h = self._ensure_handle(dev)
            rc = _cabi.lib().lsd_forward(h.ptr, visual.data_ptr(), _DTYPES[visual.dtype], _cabi.LSD_NCDHW, audio.data_ptr(), _DTYPES[audio.dtype],
                                         int(B), int(T), int(H), int(W), F_, Ta, self._precision(), logits.data_ptr(), None,
                                         workspace.data_ptr(), workspace.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)

    def workspace_bytes(self, B: int, T: int, H: int, W: int, F_: int, Ta: int) -> int:
        with self._lsd_lock:
            h = self._ensure_handle(self._device())
            need = _cabi.lib().lsd_workspace_bytes(h.ptr, int(B), int(T), int(H), int(W), int(F_), int(Ta), self._precision())
        if need == 0:
            _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
        return int(need)

    def state_generation(self) -> int:
        """Changes whenever device addresses a captured CUDA graph may hold became stale (`lsd_state_generation`)."""
        with self._lsd_lock:
            h = self._ensure_handle(self._device())
            return int(_cabi.lib().lsd_state_generation(h.ptr))

    @torch.no_grad()
    def predict(self, visual: Tensor, audio: Tensor) -> Tensor:
        self.eval()
        return self.forward(visual, audio)

    # ------------------------------------------------------------------ sub-paths (tensor-core route)
    def encode_audio(self, audio: Tensor) -> Tensor:
        """`AudioEncoder.forward` (audio_encoder.py:173-205) alone: log-mel `(B,1,F,T_a)` -> `(B, 256, T_a')` fp32."""
        if audio.dim() != 4 or audio.shape[1] != 1:
            raise ValueError(f"AudioEncoder expected input of shape (B, 1, F, T), got {tuple(audio.shape)}")
        dev = self._device()
        if audio.device != dev or audio.dtype not in _DTYPES or audio.dtype == torch.uint8:
            raise RuntimeError(f"audio must be a float tensor on {dev}")
        B, F_, Ta = int(audio.shape[0]), int(audio.shape[2]), int(audio.shape[3])
        with self._lsd_lock:
            h = self._ensure_handle(dev)
            L = _cabi.lib()
            tok = L.lsd_audio_tokens(Ta)
            out = torch.empty(B, tok, 256, dtype=torch.float32, device=dev)
            if B == 0:
                return out.transpose(1, 2)
            need = L.lsd_audio_encoder_workspace_bytes(h.ptr, B, F_, Ta)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            ws = self._workspace(need, dev)
            audio = audio.contiguous()
            rc = L.lsd_audio_encoder(h.ptr, audio.data_ptr(), _DTYPES[audio.dtype], B, F_, Ta, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                     torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return out.transpose(1, 2)

    def fuse_tokens(self, v_emb: Tensor, a_emb: Tensor) -> Tuple[Tensor, Tensor]:
        """`CrossModalAttention.forward` + `TemporalTransformer.forward` (fusion_module.py:54-87, temporal.py:79-111):
        projected embeddings `(B,T,256)`, `(B,T_a,256)` -> `(fused (B,T,256), cls (B,256))`, fp32."""
        if v_emb.dim() != 3 or a_emb.dim() != 3 or v_emb.shape[2] != 256 or a_emb.shape[2] != 256 or v_emb.shape[0] != a_emb.shape[0]:
            raise ValueError(f"expected v_emb (B,T,256) and a_emb (B,T_a,256), got {tuple(v_emb.shape)}, {tuple(a_emb.shape)}")
        dev = self._device()
        if v_emb.device != dev or a_emb.device != dev:
            raise RuntimeError(f"inputs must live on the module's device {dev}")
        B, T, TA = int(v_emb.shape[0]), int(v_emb.shape[1]), int(a_emb.shape[1])
        v_emb = v_emb.to(torch.float32).contiguous()
        a_emb = a_emb.to(torch.float32).contiguous()
        fused = torch.empty(B, T, 256, dtype=torch.float32, device=dev)
        cls = torch.empty(B, 256, dtype=torch.float32, device=dev)
        if B == 0:
            return fused, cls
        with self._lsd_lock:
            h = self._ensure_handle(dev)
            L = _cabi.lib()
            need = L.lsd_token_path_workspace_bytes(h.ptr, B, T, TA)
            if need == 0:
                _cabi.check(h.ptr, _cabi.LSD_ERR_SHAPE)
            ws = self._workspace(need, dev)
            rc = L.lsd_token_path(h.ptr, v_emb.data_ptr(), a_emb.data_ptr(), B, T, TA, fused.data_ptr(), cls.data_ptr(), ws.data_ptr(),
                                  ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(h.ptr, rc)
        return fused, cls

    # ------------------------------------------------------------------ introspection (tests / profiling)
    def stage(self, name: str) -> Tensor:
        """Flat fp32/bf16 view of a named intermediate of the last forward (lives in the workspace)."""
        h = self._lsd_handle
        off, numel, dt = C.c_size_t(), C.c_int64(), C.c_int()
        _cabi.check(h.ptr, _cabi.lib().lsd_stage_info(h.ptr, name.encode(), C.byref(off), C.byref(numel), C.byref(dt)))
        tdt = torch.float32 if dt.value == _cabi.LSD_F32 else torch.bfloat16
        esz = 4 if dt.value == _cabi.LSD_F32 else 2
        return self._lsd_ws[off.value: off.value + numel.value * esz].view(tdt)

    def planar_stage(self, name: str, shape, lo: Optional[str] = None) -> Tensor:
        """fp32 channels-last copy `(N, T, H, W, C)` of a planar bf16 activation buffer of the last tensor-core forward
        (`lsd_planar_stage_read`); H, W: the map's true full-resolution extent, whatever the buffer's layout (plain, parity-split
        or folded); `lo`: name of the low part of a (hi, lo) pair."""
        h = self._lsd_handle
        out = torch.empty(tuple(int(x) for x in shape), dtype=torch.float32, device=self._lsd_ws.device)
        rc = _cabi.lib().lsd_planar_stage_read(h.ptr, name.encode(), lo.encode() if lo else None, self._lsd_ws.data_ptr(), out.data_ptr(),
                                               out.numel(), int(shape[2]), int(shape[3]), torch.cuda.current_stream(out.device).cuda_stream)
        _cabi.check(h.ptr, rc)
        return out

    def stage_names(self):
        h = self._lsd_handle
        L = _cabi.lib()
        return [L.lsd_stage_name(h.ptr, i).decode() for i in range(L.lsd_stage_count(h.ptr))]

    def profile_enable(self, cls: int) -> None:
        """Bracket every launch of one kernel class with CUDA events (bench.py roofline):
        0 off, 1 fp32 conv kernel, 2 tcgen05 conv kernel."""
        _cabi.check(self._lsd_handle.ptr, _cabi.lib().lsd_profile_enable(self._lsd_handle.ptr, int(cls)))

    def profile_get(self):
        """-> (summed kernel ms, launches, algorithmic FLOPs) since the last call; synchronises."""
        ms, n, fl = C.c_double(), C.c_int64(), C.c_double()
        _cabi.check(self._lsd_handle.ptr, _cabi.lib().lsd_profile_get(self._lsd_handle.ptr, C.byref(ms), C.byref(n), C.byref(fl)))
        return ms.value, n.value, fl.value

    def launch_count(self) -> int:
        return self._lsd_handle.launch_count() if self._lsd_handle is not None else 0
