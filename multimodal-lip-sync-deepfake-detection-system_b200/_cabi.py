"""ctypes binding of `liblsd_b200.so` (C-ABI declared in `include/lsd_b200.h`).

The library is the product: there is no Python/torch fallback for any numeric op.  Importing this module
does not need a GPU; `lib()` raises if the shared library has not been built, and `lsd_create` fails on a
machine without an sm_100 device.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

LIB_NAME = "liblsd_b200.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

# enums of include/lsd_b200.h
LSD_OK, LSD_ERR_SHAPE, LSD_ERR_ARG, LSD_ERR_WEIGHTS, LSD_ERR_CUDA, LSD_ERR_WORKSPACE, LSD_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
LSD_F32, LSD_F16, LSD_BF16, LSD_U8, LSD_I64 = 0, 1, 2, 3, 4
LSD_NCDHW, LSD_NDHWC = 0, 1
LSD_PREC_FP32, LSD_PREC_BF16 = 0, 1
LSD_MAX_AUDIO_VARIANTS = 64
LSD_MAX_OCCLUSIONS = 1024
LSD_MAX_AUDIO_OCCLUSIONS = LSD_MAX_AUDIO_VARIANTS
LSD_MAX_WARPS = 64
LSD_JPEG_NONE, LSD_JPEG_444, LSD_JPEG_420 = 0, 1, 2
LSD_MAX_JPEG_VARIANTS = 64
LSD_RGB, LSD_BGR = 0, 1
LSD_MAX_RESIZE_VARIANTS = 64
LSD_RETIME_ONE = 32768
LSD_MAX_RETIMES = 64
LSD_AD_REVERB, LSD_AD_NOISE, LSD_AD_CLIP, LSD_AD_BAND, LSD_AD_MULAW = 1, 2, 4, 8, 16
LSD_MAX_AUDIO_DEGRADATIONS = LSD_MAX_AUDIO_VARIANTS
LSD_BRANCHES = 4
LSD_BRANCH_FEATURES = 448
LSD_MAX_BACKGROUND = 256

# every symbol include/lsd_b200.h declares (checked by tests/test_cabi.py)
EXPORTS = [
    "lsd_create", "lsd_destroy", "lsd_last_error", "lsd_version", "lsd_load_weights", "lsd_audio_tokens",
    "lsd_workspace_bytes", "lsd_forward", "lsd_logmel_frames", "lsd_logmel", "lsd_score_workspace_bytes",
    "lsd_score_windows", "lsd_stage_info", "lsd_stage_count", "lsd_stage_name", "lsd_launch_count",
    "lsd_profile_enable", "lsd_profile_get",
    "lsd_audio_encoder_workspace_bytes", "lsd_audio_encoder", "lsd_token_path_workspace_bytes", "lsd_token_path",
    "lsd_track_motion", "lsd_speech_stats", "lsd_vad_frames", "lsd_frame_energy", "lsd_vad_mask",
    "lsd_workspace_invalidate", "lsd_planar_stage_read", "lsd_state_generation", "lsd_host_pack_u8_exact", "lsd_host_pack_u8_begin", "lsd_host_pack_u8_end", "lsd_host_pack_last_ms", "lsd_expand_u8",
    "lsd_forward_audio_variants_workspace_bytes", "lsd_forward_audio_variants", "lsd_score_offsets_workspace_bytes", "lsd_score_offsets",
    "lsd_score_occlusions_workspace_bytes", "lsd_score_occlusions",
    "lsd_score_audio_occlusions_workspace_bytes", "lsd_score_audio_occlusions",
    "lsd_score_warps_workspace_bytes", "lsd_score_warps", "lsd_warp_windows_workspace_bytes", "lsd_warp_windows",
    "lsd_score_jpeg_workspace_bytes", "lsd_score_jpeg", "lsd_jpeg_windows_workspace_bytes", "lsd_jpeg_windows",
    "lsd_score_resizes_workspace_bytes", "lsd_score_resizes", "lsd_resize_tables", "lsd_resize_windows_workspace_bytes", "lsd_resize_windows",
    "lsd_score_retimes_workspace_bytes", "lsd_score_retimes", "lsd_retime_windows_workspace_bytes", "lsd_retime_windows",
    "lsd_degrade_audio_workspace_bytes", "lsd_degrade_audio", "lsd_score_audio_clips_workspace_bytes", "lsd_score_audio_clips",
    "lsd_score_branch_features", "lsd_branch_attribution_workspace_bytes", "lsd_branch_attribution",
]


class LsdTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("dtype", C.c_int), ("ndim", C.c_int), ("shape", C.c_int64 * 8), ("data", C.c_void_p)]


class LsdOcclusion(C.Structure):
    """One occlusion box in window coordinates: frames [t0,t1) x rows [y0,y1) x columns [x0,x1), filled from frame `src` of the
    un-occluded window (src >= 0) or with the call's fill value (src = -1)."""
    _fields_ = [(f, C.c_int32) for f in ("t0", "t1", "y0", "y1", "x0", "x1", "src")]


class LsdAudioOcclusion(C.Structure):
    """One audio occlusion box in window coordinates: mel columns [c0,c1) x mel bins [f0,f1) of the window's (F, Ta) log-mel
    slice, set to the call's fill value."""
    _fields_ = [(f, C.c_int32) for f in ("c0", "c1", "f0", "f1")]


class LsdWarp(C.Structure):
    """One re-crop: cv2's forward 2x3 affine matrix (src -> dst), row-major, as `cv2.warpAffine` and `cv2.getRotationMatrix2D`
    use it."""
    _fields_ = [("m", C.c_double * 6)]


class LsdJpeg(C.Structure):
    """One recompression: baseline JPEG quality 1..100 and chroma sampling (LSD_JPEG_420 / LSD_JPEG_444; LSD_JPEG_NONE copies)."""
    _fields_ = [("quality", C.c_int32), ("sampling", C.c_int32)]


class LsdResize(C.Structure):
    """One face size (h, w): every frame down to it with cv2's INTER_AREA and back to the crop size with INTER_LINEAR; the crop
    size itself copies the frame."""
    _fields_ = [("h", C.c_int32), ("w", C.c_int32)]


class LsdRetime(C.Structure):
    """One output frame of a retimed window: up to four taps, frame offsets `src` from the window's first track frame (clamped to the
    track) and Q15 weights >= 0 summing to LSD_RETIME_ONE."""
    _fields_ = [("src", C.c_int32 * 4), ("weight", C.c_int32 * 4)]


class LsdAudioDegradation(C.Structure):
    """One audio degradation: the `stages` bits (LSD_AD_*) and the parameters of the stages they enable: reverb time rt60 (s), noise
    SNR (dB), overdrive gain (dB), band rate (8000 or 4000 Hz) and the generator's seed."""
    _fields_ = [("stages", C.c_int32), ("rt60", C.c_float), ("snr_db", C.c_float), ("gain_db", C.c_float), ("band_rate", C.c_int32),
                ("seed", C.c_uint32)]


class LsdAux(C.Structure):
    _fields_ = [("visual_tokens", C.c_void_p), ("audio_tokens", C.c_void_p), ("fused_tokens", C.c_void_p), ("cls_output", C.c_void_p)]


_lib = None
_lock = threading.Lock()


def lib() -> C.CDLL:
    """Load the shared library once; fail loudly when it is missing (no fallback path exists)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_NAME} is not built ({LIB_PATH}); run `python -c 'import __graft_entry__ as g; g.build()'` "
                "from the repo root.  There is no CPU/torch fallback for the window-scoring path.")
        L = C.CDLL(LIB_PATH)
        vp, i, sz, i64 = C.c_void_p, C.c_int, C.c_size_t, C.c_int64
        L.lsd_create.argtypes = [C.POINTER(vp), i]; L.lsd_create.restype = i
        L.lsd_destroy.argtypes = [vp]; L.lsd_destroy.restype = None
        L.lsd_last_error.argtypes = [vp]; L.lsd_last_error.restype = C.c_char_p
        L.lsd_version.argtypes = []; L.lsd_version.restype = i
        L.lsd_load_weights.argtypes = [vp, C.POINTER(LsdTensor), i]; L.lsd_load_weights.restype = i
        L.lsd_audio_tokens.argtypes = [i]; L.lsd_audio_tokens.restype = i
        L.lsd_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i]; L.lsd_workspace_bytes.restype = sz
        L.lsd_forward.argtypes = [vp, vp, i, i, vp, i, i, i, i, i, i, i, i, vp, C.POINTER(LsdAux), vp, sz, vp]
        L.lsd_forward.restype = i
        L.lsd_logmel_frames.argtypes = [i64]; L.lsd_logmel_frames.restype = i
        L.lsd_logmel.argtypes = [vp, vp, C.POINTER(i64), i, vp, C.POINTER(i64), vp, vp]; L.lsd_logmel.restype = i
        L.lsd_score_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i]; L.lsd_score_workspace_bytes.restype = sz
        L.lsd_score_windows.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i, i, i, vp, vp, sz, vp]
        L.lsd_score_windows.restype = i
        L.lsd_stage_info.argtypes = [vp, C.c_char_p, C.POINTER(sz), C.POINTER(i64), C.POINTER(i)]; L.lsd_stage_info.restype = i
        L.lsd_stage_count.argtypes = [vp]; L.lsd_stage_count.restype = i
        L.lsd_stage_name.argtypes = [vp, i]; L.lsd_stage_name.restype = C.c_char_p
        L.lsd_launch_count.argtypes = [vp]; L.lsd_launch_count.restype = i64
        L.lsd_profile_enable.argtypes = [vp, i]; L.lsd_profile_enable.restype = i
        L.lsd_profile_get.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i64), C.POINTER(C.c_double)]; L.lsd_profile_get.restype = i
        L.lsd_audio_encoder_workspace_bytes.argtypes = [vp, i, i, i]; L.lsd_audio_encoder_workspace_bytes.restype = sz
        L.lsd_audio_encoder.argtypes = [vp, vp, i, i, i, i, vp, vp, sz, vp]; L.lsd_audio_encoder.restype = i
        L.lsd_token_path_workspace_bytes.argtypes = [vp, i, i, i]; L.lsd_token_path_workspace_bytes.restype = sz
        L.lsd_token_path.argtypes = [vp, vp, vp, i, i, i, vp, vp, vp, sz, vp]; L.lsd_token_path.restype = i
        L.lsd_track_motion.argtypes = [vp, vp, i, i, i, i, i, vp, vp, vp]; L.lsd_track_motion.restype = i
        L.lsd_speech_stats.argtypes = [vp, vp, vp, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i, vp, vp, vp, vp, vp]
        L.lsd_speech_stats.restype = i
        L.lsd_vad_frames.argtypes = [i64]; L.lsd_vad_frames.restype = i
        L.lsd_frame_energy.argtypes = [vp, vp, i64, vp, vp]; L.lsd_frame_energy.restype = i
        L.lsd_vad_mask.argtypes = [vp, vp, i, C.c_float, vp, vp]; L.lsd_vad_mask.restype = i
        L.lsd_workspace_invalidate.argtypes = [vp]; L.lsd_workspace_invalidate.restype = i
        L.lsd_state_generation.argtypes = [vp]; L.lsd_state_generation.restype = i64
        L.lsd_host_pack_u8_exact.argtypes = [vp, vp, i64, i]; L.lsd_host_pack_u8_exact.restype = i
        L.lsd_host_pack_u8_begin.argtypes = [vp, vp, i64, i]; L.lsd_host_pack_u8_begin.restype = i
        L.lsd_host_pack_u8_end.argtypes = []; L.lsd_host_pack_u8_end.restype = i
        L.lsd_host_pack_last_ms.argtypes = []; L.lsd_host_pack_last_ms.restype = C.c_double
        L.lsd_expand_u8.argtypes = [vp, vp, i64, vp]; L.lsd_expand_u8.restype = i
        L.lsd_planar_stage_read.argtypes = [vp, C.c_char_p, C.c_char_p, vp, vp, i64, i, i, vp]; L.lsd_planar_stage_read.restype = i
        L.lsd_forward_audio_variants_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i, i]; L.lsd_forward_audio_variants_workspace_bytes.restype = sz
        L.lsd_forward_audio_variants.argtypes = [vp, vp, i, i, vp, i, i, i, i, i, i, i, i, i, vp, vp, sz, vp]
        L.lsd_forward_audio_variants.restype = i
        L.lsd_score_offsets_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i, i]; L.lsd_score_offsets_workspace_bytes.restype = sz
        L.lsd_score_offsets.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i,
                                        C.POINTER(C.c_int32), i, i, i, vp, C.POINTER(C.c_int32), vp, sz, vp]
        L.lsd_score_offsets.restype = i
        L.lsd_score_occlusions_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i]; L.lsd_score_occlusions_workspace_bytes.restype = sz
        L.lsd_score_occlusions.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i,
                                           C.POINTER(LsdOcclusion), i, i, i, i, vp, vp, sz, vp]
        L.lsd_score_occlusions.restype = i
        L.lsd_score_audio_occlusions_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i, i]
        L.lsd_score_audio_occlusions_workspace_bytes.restype = sz
        L.lsd_score_audio_occlusions.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i,
                                                 C.POINTER(LsdAudioOcclusion), i, C.c_float, i, i, vp, vp, sz, vp]
        L.lsd_score_audio_occlusions.restype = i
        L.lsd_score_warps_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i, i]; L.lsd_score_warps_workspace_bytes.restype = sz
        L.lsd_score_warps.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i,
                                      C.POINTER(LsdWarp), i, i, i, vp, vp, sz, vp]
        L.lsd_score_warps.restype = i
        L.lsd_warp_windows_workspace_bytes.argtypes = [i, i, i, i, i]; L.lsd_warp_windows_workspace_bytes.restype = sz
        L.lsd_warp_windows.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), i, i, C.POINTER(LsdWarp), i, vp, vp, sz, vp]
        L.lsd_warp_windows.restype = i
        L.lsd_score_jpeg_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i, i]; L.lsd_score_jpeg_workspace_bytes.restype = sz
        L.lsd_score_jpeg.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i,
                                     C.POINTER(LsdJpeg), i, i, i, i, vp, vp, sz, vp]
        L.lsd_score_jpeg.restype = i
        L.lsd_jpeg_windows_workspace_bytes.argtypes = [i, i, i, i, i]; L.lsd_jpeg_windows_workspace_bytes.restype = sz
        L.lsd_jpeg_windows.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), i, i, C.POINTER(LsdJpeg), i, i, vp, vp, sz, vp]
        L.lsd_jpeg_windows.restype = i
        L.lsd_score_resizes_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i, i]; L.lsd_score_resizes_workspace_bytes.restype = sz
        L.lsd_score_resizes.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i,
                                        C.POINTER(LsdResize), i, i, i, vp, vp, sz, vp]
        L.lsd_score_resizes.restype = i
        L.lsd_resize_tables.argtypes = [C.POINTER(LsdResize), i, i, i, vp]; L.lsd_resize_tables.restype = i64
        L.lsd_resize_windows_workspace_bytes.argtypes = [i, i, i, i, i]; L.lsd_resize_windows_workspace_bytes.restype = sz
        L.lsd_resize_windows.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), i, i, C.POINTER(LsdResize), i, vp, vp, sz, vp]
        L.lsd_resize_windows.restype = i
        L.lsd_score_retimes_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i, i]; L.lsd_score_retimes_workspace_bytes.restype = sz
        L.lsd_score_retimes.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i,
                                        C.POINTER(LsdRetime), i, i, i, vp, vp, sz, vp]
        L.lsd_score_retimes.restype = i
        L.lsd_retime_windows_workspace_bytes.argtypes = [i, i, i, i, i]; L.lsd_retime_windows_workspace_bytes.restype = sz
        L.lsd_retime_windows.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), i, i, C.POINTER(LsdRetime), i, vp, vp, sz, vp]
        L.lsd_retime_windows.restype = i
        L.lsd_score_branch_features.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i, i, i,
                                                vp, vp, vp, sz, vp]
        L.lsd_score_branch_features.restype = i
        L.lsd_branch_attribution_workspace_bytes.argtypes = [i, i]; L.lsd_branch_attribution_workspace_bytes.restype = sz
        L.lsd_branch_attribution.argtypes = [vp, vp, i, vp, i, vp, vp, vp, sz, vp]; L.lsd_branch_attribution.restype = i
        L.lsd_degrade_audio_workspace_bytes.argtypes = [i64, i]; L.lsd_degrade_audio_workspace_bytes.restype = sz
        L.lsd_degrade_audio.argtypes = [vp, vp, i64, C.POINTER(LsdAudioDegradation), i, vp, vp, sz, vp]; L.lsd_degrade_audio.restype = i
        L.lsd_score_audio_clips_workspace_bytes.argtypes = [vp, i, i, i, i, i, i, i, i]; L.lsd_score_audio_clips_workspace_bytes.restype = sz
        L.lsd_score_audio_clips.argtypes = [vp, vp, i, i, i, C.POINTER(C.c_int32), C.POINTER(C.c_int32), i, i, vp, i, i, i, i, i, i, i,
                                            vp, vp, sz, vp]
        L.lsd_score_audio_clips.restype = i
        _lib = L
        return L


def check(handle, rc: int) -> None:
    """Map a C status to the reference's error convention: shape errors -> ValueError (HTTP 400 in
    app/api/routes.py:46-48), everything else -> RuntimeError."""
    if rc == LSD_OK:
        return
    msg = lib().lsd_last_error(handle)
    text = msg.decode("utf-8", "replace") if msg else f"lsd error {rc}"
    if rc == LSD_ERR_SHAPE:
        raise ValueError(text)
    raise RuntimeError(text)


class Handle:
    """Owns one `lsd_handle*` (one per model instance and device); not thread-safe — callers hold `self.lock`."""

    def __init__(self, device_index: int):
        self.lock = threading.RLock()
        self.ptr = C.c_void_p()
        rc = lib().lsd_create(C.byref(self.ptr), int(device_index))
        if rc != LSD_OK:
            msg = lib().lsd_last_error(None)
            raise RuntimeError(msg.decode("utf-8", "replace") if msg else f"lsd_create failed ({rc})")
        self.device_index = int(device_index)

    def close(self) -> None:
        if self.ptr:
            lib().lsd_destroy(self.ptr)
            self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def launch_count(self) -> int:
        return int(lib().lsd_launch_count(self.ptr))
