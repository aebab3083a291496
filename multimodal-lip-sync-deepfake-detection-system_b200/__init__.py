"""B200-native window scoring for the R2Plus1D-Sync lip-sync detector (hot path only).

Public surface mirrors the reference (`app/models/lip_sync_model.py`, `app/inference/predictor.py`,
`app/preprocessing/audio.py`) for the window-scoring path; every numeric op runs in the hand-written
sm_100a CUDA library `csrc/` through its C-ABI (`include/lsd_b200.h`).  There is no CPU fallback.
"""
from .state_spec import state_spec, make_synthetic_state_dict, synthetic_windows, BUFFER_SUFFIXES  # noqa: F401
from .model import LipSyncModel  # noqa: F401
from .inference import Predictor, partition_windows, gather_logits  # noqa: F401
from .aggregate import aggregate_long_video, select_windows_by_time, frame_evidence_timeline, columns_to_frames, augmentation_stability  # noqa: F401
from .long_video import predict_long_video_from_tracks  # noqa: F401
from .validate import run_preprocessed_validation, compute_metrics  # noqa: F401
from .audio import preprocess_audio, preprocess_audio_pcm, logmel_db, fit_frames, detect_voice_activity_pcm  # noqa: F401

__all__ = ["state_spec", "make_synthetic_state_dict", "synthetic_windows", "LipSyncModel", "Predictor",
           "partition_windows", "gather_logits", "aggregate_long_video", "select_windows_by_time", "predict_long_video_from_tracks", "run_preprocessed_validation", "compute_metrics", "preprocess_audio", "preprocess_audio_pcm", "logmel_db", "fit_frames", "detect_voice_activity_pcm"]
