/*
 * lsd_b200.h — C-ABI of the B200-native window-scoring library (liblsd_b200.so).
 *
 * The reference (PRADUMAN-KR/Multimodal-Lip-Sync-Deepfake-Detection-System) is 100 % Python and has no
 * FFI of its own (SURVEY.md §8b); its boundary for this path is
 *   - `LipSyncModel.forward(visual, audio) -> logits`      app/models/lip_sync_model.py:86-136
 *   - `LipSyncModel.load_state_dict(state, strict=True)`   app/inference/predictor.py:187-194
 *   - `preprocess_audio(...)` (librosa log-mel)            app/preprocessing/audio.py:47-102
 *   - `Predictor._run_chunked_inference(...)`              app/inference/predictor.py:554-580
 *   - `Predictor._align_audio_chunk(...)`                  app/inference/predictor.py:525-552
 * Each entry point below names the reference interface it replaces.  The Python host layer
 * (`lipsync_b200`) binds these with ctypes; INTEGRATION.md shows the stub a reference maintainer adds.
 *
 * Conventions: plain pointers and sizes only (no torch types).  Every function returns 0 on success
 * or a negative lsd_status; the message is available from lsd_last_error().  LSD_ERR_SHAPE maps to
 * Python ValueError (HTTP 400 in the reference, app/api/routes.py:46-48), everything else to
 * RuntimeError.  All device pointers are caller-owned; work is enqueued asynchronously on `stream`
 * (a cudaStream_t passed as void*), with no hidden synchronisation and no hidden device allocation in
 * lsd_forward / lsd_logmel / lsd_score_windows (the caller provides the workspace).  A handle is not
 * thread-safe; the Python layer serialises access with a lock (the reference can enter forward from
 * two threads, SURVEY.md §8b).
 */
#ifndef LSD_B200_H
#define LSD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lsd_handle lsd_handle;

typedef enum {
  LSD_OK = 0,
  LSD_ERR_SHAPE = -1,      /* wrong rank / extent            -> ValueError   */
  LSD_ERR_ARG = -2,        /* null pointer, bad enum         -> RuntimeError */
  LSD_ERR_WEIGHTS = -3,    /* missing / mis-shaped state_dict entry (strict) */
  LSD_ERR_CUDA = -4,       /* CUDA runtime / driver error                    */
  LSD_ERR_WORKSPACE = -5,  /* workspace too small                            */
  LSD_ERR_UNSUPPORTED = -6 /* e.g. not an sm_100 device                      */
} lsd_status;

typedef enum { LSD_F32 = 0, LSD_F16 = 1, LSD_BF16 = 2, LSD_U8 = 3, LSD_I64 = 4 } lsd_dtype;

/* video memory layout: NCDHW is what the reference hands over (video.py:552-556 builds (3,T,H,W));
 * NDHWC is the raw-track layout (N,T,H,W,3) that the window builder produces. */
typedef enum { LSD_NCDHW = 0, LSD_NDHWC = 1 } lsd_layout;

/* arithmetic of the conv/GEMM stack: FP32 = CUDA-core FFMA path (parity <= 1e-4 rel);
 * BF16 = tcgen05 tensor-core path with fp32 accumulation (parity <= 2e-2 abs on logits). */
typedef enum { LSD_PREC_FP32 = 0, LSD_PREC_BF16 = 1 } lsd_precision;

/* One state_dict entry, host memory (replaces torch.load + load_state_dict, predictor.py:187-194). */
typedef struct {
  const char* name;   /* reference key, e.g. "visual_encoder.layer1.conv1.0.weight" */
  int dtype;          /* LSD_F32 (all parameters/buffers) or LSD_I64 (num_batches_tracked, ignored) */
  int ndim;
  int64_t shape[8];
  const void* data;   /* host pointer, contiguous */
} lsd_tensor;

/* Optional extra outputs of lsd_forward (the `return_aux=True` dict, lip_sync_model.py:130-136).
 * Any pointer may be NULL.  All fp32, device memory. */
typedef struct {
  float* visual_tokens; /* (B, T, 256)        */
  float* audio_tokens;  /* (B, T_audio_tok, 256), T_audio_tok = lsd_audio_tokens(Ta) */
  float* fused_tokens;  /* (B, T, 256)        */
  float* cls_output;    /* (B, 256)           */
} lsd_aux;

/* ---- lifetime ------------------------------------------------------------------------------ */
int lsd_create(lsd_handle** out, int device);
void lsd_destroy(lsd_handle* h);
const char* lsd_last_error(lsd_handle* h); /* h may be NULL: returns the last create() error */
int lsd_version(void);

/* ---- weights: replaces LipSyncModel.load_state_dict(strict=True) ----------------------------- */
/* Consumes the 270-entry reference state_dict (fp32, host), folds eval-mode BatchNorm (+conv bias)
 * into per-channel scale/shift (SURVEY.md App. A) and repacks every conv/linear weight into the
 * device layouts the kernels read (fp32 [tap][Cin][Cout]; bf16 UMMA core-matrix tiles). */
int lsd_load_weights(lsd_handle* h, const lsd_tensor* tensors, int n);

/* ---- forward: replaces LipSyncModel.forward(visual, audio) ----------------------------------- */
int lsd_audio_tokens(int Ta);     /* audio token count produced by the audio encoder for Ta mel frames */
size_t lsd_workspace_bytes(lsd_handle* h, int B, int T, int H, int W, int F, int Ta, int precision);
int lsd_forward(lsd_handle* h,
                const void* video, int video_dtype, int video_layout, /* device, (B,3,T,H,W) or (B,T,H,W,3) */
                const void* audio, int audio_dtype,                   /* device, (B,1,F,Ta) */
                int B, int T, int H, int W, int F, int Ta,
                int precision,
                float* logits_out,                                    /* device, B floats */
                const lsd_aux* aux_or_null,
                void* workspace, size_t workspace_bytes,
                void* stream);

/* Workspace contract (tensor-core route): the zero padding of the planar activation buffers is written once per
 * (workspace pointer, size, shapes) and then kept inside the workspace between calls — the library remembers the last
 * workspace it initialised and skips the memset when the same one comes back.  The caller must therefore not modify the
 * workspace between calls that reuse it; after writing into it, or after freeing it (a later allocation may return the
 * same address), call lsd_workspace_invalidate() before the next forward.  Calls through the library itself (other
 * shapes, the fp32 route, lsd_score_windows halves) are tracked internally. */
int lsd_workspace_invalidate(lsd_handle* h);

/* ---- sub-paths of the forward (tensor-core route; same kernels and numerics as inside lsd_forward) ------- */
/* AudioEncoder.forward (app/models/audio_encoder.py:173-205): log-mel windows (B,1,F,Ta), device, any float dtype
 * -> feats_out (B, lsd_audio_tokens(Ta), 256) fp32 device rows (the reference returns the transpose (B,256,T')). */
size_t lsd_audio_encoder_workspace_bytes(lsd_handle* h, int B, int F, int Ta);
int lsd_audio_encoder(lsd_handle* h, const void* audio, int audio_dtype, int B, int F, int Ta, float* feats_out,
                      void* workspace, size_t workspace_bytes, void* stream);
/* CrossModalAttention.forward (app/models/fusion_module.py:54-87) followed by TemporalTransformer.forward
 * (app/models/temporal.py:79-111): projected embeddings v_emb (B,T,256), a_emb (B,Ta_tokens,256), fp32 device
 * -> fused_out (B,T,256) and/or cls_out (B,256), fp32 device (either may be NULL).  Same kernels as inside lsd_forward; the
 * full forward feeds them the cross-attention in-projections from a GEMM merged with FeatureProjection, this entry point
 * computes them from the embeddings, so the two agree to ~1e-4 relative, not bit for bit. */
size_t lsd_token_path_workspace_bytes(lsd_handle* h, int B, int T, int Ta_tokens);
int lsd_token_path(lsd_handle* h, const float* v_emb, const float* a_emb, int B, int T, int Ta_tokens,
                   float* fused_out, float* cls_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- log-mel front end: replaces preprocess_audio's librosa calls (audio.py:80-91) ----------- */
/* pcm: device fp32 mono 16 kHz, clips concatenated; clip c spans [clip_offsets[c], clip_offsets[c+1]).
 * mel_out: device fp32, clip c written as (80, frames_c) row-major at mel_offsets[c] (in floats),
 * frames_c = 1 + len_c / 160.  ref=max is per clip (two-pass).  scratch: n_clips floats (device). */
int lsd_logmel_frames(int64_t n_samples);
int lsd_logmel(lsd_handle* h, const float* pcm, const int64_t* clip_offsets_host, int n_clips,
               float* mel_out, const int64_t* mel_offsets_host, float* scratch, void* stream);

/* ---- window builder + batched scoring: replaces the serial loop of _run_chunked_inference ---- */
/* track: device uint8 (n_frames, H, W, 3) mouth crops (video.py:576-588 contract, before the
 * astype(float32)/255 of video.py:552-556).  starts: host int32 absolute start frame per window,
 * relative to track frame 0.  mel_full: device fp32 (1, F, Ta_full) clip-level log-mel.
 * Audio windows follow _align_audio_chunk (predictor.py:525-552) with chunk_a_size = Ta.
 * Builds the windows on device and runs lsd_forward in batches of `batch`. */
size_t lsd_score_workspace_bytes(lsd_handle* h, int batch, int T, int H, int W, int F, int Ta, int precision);
/* Passing a workspace of at least TWICE lsd_score_workspace_bytes() lets lsd_score_windows (tensor-core route, more than one
 * batch) alternate batches between its two halves and overlap the latency-bound tail of batch k (audio encoder, token path,
 * head, artifact branch: internal streams) with the visual encoder of batch k+1; results are bit-identical either way. */
int lsd_score_windows(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W,
                      const int32_t* starts_host, const int32_t* audio_starts_host_or_null, int n_windows, int T,
                      const float* mel_full, int F, int Ta_full, int total_v_frames, int Ta,
                      int precision, int batch, float* logits_out,
                      void* workspace, size_t workspace_bytes, void* stream);
/* audio_starts_host_or_null: explicit first mel column per window (clamped like _align_audio_chunk).  A rank that holds
 * only its own span of a sharded track passes span-relative `starts` and the audio starts computed from the absolute frame
 * indices (SURVEY.md §8e); NULL = computed here from `starts` as predictor.py:540-547 does. */

/* ---- audio-offset sweep: one visual-encoder pass, K audio windows per video ------------------------------------ */
/* The reference trains with torch.roll-shifted audio as sync negatives (train.py:169-182), so its logit as a function of the
 * audio offset is a sync profile: a real clip with a constant A/V delay peaks away from offset 0, a lip-sync fake has no clear
 * peak.  Scoring K audio windows against one video this way repeats only the audio-dependent part of LipSyncModel.forward
 * (lip_sync_model.py:86-136): the audio encoder, the cross-modal attention + temporal transformer and the classifier head.  The
 * visual encoder and the artifact branch run once per video.
 * The logit of (b, k) is bit for bit what lsd_forward gives video b with audio window k (same precision).  The tensor-core route
 * with the fused token kernels shares the video side; every other configuration (fp32, the launch-by-launch token path) runs one
 * lsd_forward per audio window, with the same results. */
#define LSD_MAX_AUDIO_VARIANTS 64
/* video as in lsd_forward; audio: device (B,K,1,F,Ta), window k of video b at row b*K + k; logits_out: device (B,K) fp32.
 * LSD_ERR_SHAPE for K < 1 or K > LSD_MAX_AUDIO_VARIANTS. */
size_t lsd_forward_audio_variants_workspace_bytes(lsd_handle* h, int B, int K, int T, int H, int W, int F, int Ta, int precision);
int lsd_forward_audio_variants(lsd_handle* h, const void* video, int video_dtype, int video_layout,
                               const void* audio, int audio_dtype,
                               int B, int K, int T, int H, int W, int F, int Ta, int precision,
                               float* logits_out, void* workspace, size_t workspace_bytes, void* stream);
/* lsd_score_windows with K audio offsets per window (Predictor._align_audio_chunk, predictor.py:525-552, moved by whole mel
 * columns).  offsets_host: K int32 offsets d in mel columns (10 ms; d > 0 = the audio slice starts later).  Window i with base
 * audio start a_i (computed, or audio_starts_host_or_null[i], exactly as lsd_score_windows does) reads its slice for offset d
 * at clamp(a_i + d): past the end -> Ta_full - Ta, then never below 0 — the rule lsd_score_windows applies.  (i, k) is valid
 * when no clamping was needed: 0 <= a_i + d_k <= Ta_full - Ta.
 * logits_out: device (n_windows, K) fp32, entry (i, k) bit for bit lsd_score_windows for window i with the effective start
 * as its explicit audio start.  eff_audio_starts_host_or_null: host (n_windows, K) int32 effective starts, written before any
 * GPU work is enqueued.  LSD_ERR_ARG for offsets_host == NULL, LSD_ERR_SHAPE for K out of range or a window outside the track. */
size_t lsd_score_offsets_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision);
int lsd_score_offsets(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W,
                      const int32_t* starts_host, const int32_t* audio_starts_host_or_null, int n_windows, int T,
                      const float* mel_full, int F, int Ta_full, int total_v_frames, int Ta,
                      const int32_t* offsets_host, int K, int precision, int batch,
                      float* logits_out, int32_t* eff_audio_starts_host_or_null,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---- occlusion evidence: window scores with a region of the window hidden ---------------------------------- */
/* This entry has no reference counterpart.  It builds on the scoring loop of Predictor._run_chunked_inference
 * (predictor.py:554-580, lsd_score_windows): every window is scored K times, once per occlusion box, and the change of the
 * logit is that region's evidence.  A box is seven int32 values in window coordinates.  With win the un-occluded uint8 window
 * (frames starts_host[i] .. starts_host[i]+T-1 of the track), the occluded window is
 *   out[t,y,x,:] = (t0<=t<t1 && y0<=y<y1 && x0<=x<x1) ? (src < 0 ? fill : win[src,y,x,:]) : win[t,y,x,:]
 * src >= 0 copies frame src of the UN-occluded window, also when src lies inside the box.  A box with t0==t1, y0==y1 or x0==x1
 * is empty: the row is the plain window.  Typical boxes: a freeze of frames [t0,t1) (full frame, src = t0-1, or t1 when t0 == 0)
 * and a fill of a spatial cell over all frames (src = -1). */
typedef struct { int32_t t0, t1, y0, y1, x0, x1, src; } lsd_occlusion;
#define LSD_MAX_OCCLUSIONS 1024
/* Rows are (window, box) pairs in window-major order, row r = i*K + k; `batch` counts rows.  A row's audio slice is its window's
 * slice, with the base-start rule of lsd_score_windows (computed, or audio_starts_host_or_null[i], clamped).  The occluded windows
 * of a batch are built on the device (16-byte loads and stores, reading only the window's frames) and scored by the plain batch
 * path of lsd_score_windows, so logits_out (device, (n_windows, K) fp32) entry (i, k) is bit for bit lsd_score_windows on window
 * i occluded on the host, with the same audio start.  A workspace of at least twice lsd_score_occlusions_workspace_bytes enables
 * the cross-batch pipelining of lsd_score_windows; a short last batch runs in exactly the queried size.  Everything is checked
 * before any GPU work: LSD_ERR_SHAPE for K outside 1..LSD_MAX_OCCLUSIONS, a box outside [0,T]x[0,H]x[0,W] or with t0>t1
 * (likewise y, x), src outside -1..T-1, or a window outside the track; LSD_ERR_ARG for boxes == NULL or fill outside 0..255. */
size_t lsd_score_occlusions_workspace_bytes(lsd_handle* h, int batch, int T, int H, int W, int F, int Ta, int precision);
int lsd_score_occlusions(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W,
                         const int32_t* starts_host, const int32_t* audio_starts_host_or_null, int n_windows, int T,
                         const float* mel_full, int F, int Ta_full, int total_v_frames, int Ta,
                         const lsd_occlusion* boxes, int K, int fill, int precision, int batch,
                         float* logits_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- crop-jitter robustness: window scores of re-cropped windows ------------------------------------------ */
/* This entry has no reference counterpart.  The reference's mouth crops come from a CPU face tracker whose boxes move with the
 * detector that fired and jitter from frame to frame (app/preprocessing/face_detection.py, video.py:455-590); it asks whether a window's score would hold
 * had the crop been placed differently.  Every window is scored K times, once per variant.  Variant k re-crops frame t of the
 * window with its own forward 2x3 matrix (a different matrix per frame models tracker jitter):
 *   out[t] = cv2.warpAffine(win[t], M[k,t], (W, H), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)
 * bit for bit (8-bit integer arithmetic on tables built on the host exactly as cv::warpAffine builds them, including its
 * inversion of M in double).  lsd_warp is cv2's forward matrix, row-major, src -> dst: the convention of cv2.warpAffine and
 * cv2.getRotationMatrix2D. */
typedef struct { double m[6]; } lsd_warp;
#define LSD_MAX_WARPS 64
/* warps: host, K*T matrices, variant-major (warps[k*T + t]).  Rows are (window, variant) pairs in window-major order, row
 * r = i*K + k; `batch` counts rows.  A row's audio slice is its window's slice, with the base-start rule of lsd_score_windows
 * (computed, or audio_starts_host_or_null[i], clamped).  The warped windows of a batch are built on the device and scored by the
 * plain batch path of lsd_score_windows, so logits_out (device, (n_windows, K) fp32) entry (i, k) is bit for bit lsd_score_windows
 * on window i warped on the host, with the same audio start.  A workspace of at least twice lsd_score_warps_workspace_bytes enables
 * the cross-batch pipelining of lsd_score_windows; a short last batch runs in exactly the queried size.  Everything is checked
 * before any GPU work: LSD_ERR_SHAPE for K outside 1..LSD_MAX_WARPS, a window outside the track, or a matrix whose inverse maps a
 * pixel of the frame to a coordinate beyond +-32767 (cv2's int16 tap coordinates would saturate); LSD_ERR_ARG for warps == NULL,
 * a non-finite entry or a singular matrix. */
size_t lsd_score_warps_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision);
int lsd_score_warps(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W,
                    const int32_t* starts_host, const int32_t* audio_starts_host_or_null, int n_windows, int T,
                    const float* mel_full, int F, int Ta_full, int total_v_frames, int Ta,
                    const lsd_warp* warps, int K, int precision, int batch,
                    float* logits_out, void* workspace, size_t workspace_bytes, void* stream);
/* The re-cropped windows themselves, built by the same kernel lsd_score_warps scores: out (device uint8, (n_windows, K, T, H, W, 3))
 * holds window i under variant k at [i][k], each frame bit for bit the cv2.warpAffine above.  Same checks as lsd_score_warps;
 * workspace: lsd_warp_windows_workspace_bytes (the tables and the window starts). */
size_t lsd_warp_windows_workspace_bytes(int n_windows, int K, int T, int H, int W);
int lsd_warp_windows(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W,
                     const int32_t* starts_host, int n_windows, int T, const lsd_warp* warps, int K,
                     uint8_t* out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- audio occlusion evidence: window scores with a region of the window's log-mel masked ------------------ */
/* This entry has no reference counterpart.  Window i's audio slice is the (F, Ta) log-mel window of Predictor._align_audio_chunk
 * (predictor.py:525-552) that lsd_score_windows gives it: first column the base start a_i (computed, or
 * audio_starts_host_or_null[i], clamped as there), the last column of the clip repeated past its end.  A box is four int32
 * values in window coordinates, columns [c0,c1) x mel bins [f0,f1); the masked slice is
 *   out[f,c] = (c0<=c<c1 && f0<=f<f1) ? fill : win[f,c]
 * applied after the padding, so a box may cover repeated columns.  A box with c0==c1 or f0==f1 is empty: the row is the plain
 * window.  fill -80 is the floor of the library's log-mel (power_to_db(ref=max, top_db=80), logmel.cu), i.e. silence relative to
 * the clip's maximum.  Typical boxes: a time segment over all bins and a mel band over all columns. */
typedef struct { int32_t c0, c1, f0, f1; } lsd_audio_occlusion;
#define LSD_MAX_AUDIO_OCCLUSIONS LSD_MAX_AUDIO_VARIANTS
/* Rows are (window, box) pairs in window-major order, row r = i*K + k; `batch` counts windows, as in lsd_score_offsets.  The masked
 * slices of a batch are written on the device, end to end, into a pseudo clip (F, nb*K*Ta) in the workspace, and row j of the
 * batch reads columns [j*Ta, (j+1)*Ta) of it as its explicit audio start.  The tensor-core route with the fused token kernels
 * scores them with the shared-visual forward of lsd_score_offsets (visual encoder and artifact branch once per window); every
 * other configuration scores them with lsd_score_windows, each window repeated K times.  logits_out: device (n_windows, K) fp32,
 * entry (i, k) bit for bit lsd_score_windows on window i with slice k masked on the host (any such clip, explicit audio start).
 * Everything is checked before any GPU work: LSD_ERR_SHAPE for K outside 1..LSD_MAX_AUDIO_OCCLUSIONS, a box outside
 * [0,Ta]x[0,F] or with c0>c1 or f0>f1, or a window outside the track; LSD_ERR_ARG for boxes == NULL, a non-finite fill or a
 * null pointer. */
size_t lsd_score_audio_occlusions_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision);
int lsd_score_audio_occlusions(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W,
                               const int32_t* starts_host, const int32_t* audio_starts_host_or_null, int n_windows, int T,
                               const float* mel_full, int F, int Ta_full, int total_v_frames, int Ta,
                               const lsd_audio_occlusion* boxes, int K, float fill, int precision, int batch,
                               float* logits_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- speaking alignment / mouth motion: the per-window numpy loops of _predict_long_video ------------------ */
/* Frame-difference energies of a track (Predictor._speaking_alignment_score, app/inference/predictor.py:339-345, and
 * _mouth_motion_energy_check, :395-402): for every frame pair f in [0, n_frames-1)
 *   motion_full[f] = mean_{h,w} |gray[f+1]-gray[f]|,  motion_low[f] = the same over the lower half rows (h >= H/2),
 * gray = channel mean of the crop scaled to [0,1].  video: device uint8 (n_frames,H,W,3) track (LSD_U8, LSD_NDHWC) or a
 * device float32 (3,n_frames,H,W) window (LSD_F32, LSD_NCDHW: the reference's visual_np). */
int lsd_track_motion(lsd_handle* h, const void* video, int dtype, int layout, int n_frames, int H, int W,
                     float* motion_full, float* motion_low, void* stream);
/* Per window (start frame starts_host[i], T frames; audio slice as in lsd_score_windows):
 *   speaking_out[i]     = Predictor._speaking_alignment_score(window, mel slice)      predictor.py:333-370
 *   mouth_motion_out[i] = mean lower-face motion, audio_energy_out[i] = mean mel dB     predictor.py:395-402
 * (the likely_fake / uncertain / no_issue thresholds of :403-413 are applied by the host layer).
 * idx_scratch: device, 2*n_windows int32.  T, Ta <= 128. */
int lsd_speech_stats(lsd_handle* h, const float* motion_full, const float* motion_low, int n_frames,
                     const int32_t* starts_host, const int32_t* audio_starts_host_or_null, int n_windows, int T,
                     const float* mel_full, int F, int Ta_full, int total_v_frames, int Ta,
                     float* speaking_out, float* mouth_motion_out, float* audio_energy_out,
                     int32_t* idx_scratch, void* stream);

/* ---- energy VAD: the per-frame loops of detect_voice_activity (app/preprocessing/audio.py:178-230) ---------- */
/* energy_out[i] = mean(y[160 i : min(160 i + 400, n)]^2) for i < lsd_vad_frames(n) = ceil(n / 160)   (audio.py:182-192);
 * mask_out[i] = OR_{j in [i-1,i+1]} (energy[j] >= threshold)                                         (audio.py:214-221).
 * The threshold (median / 20th percentile / torchaudio VAD energy, audio.py:196-212) is computed by the host layer. */
int lsd_vad_frames(int64_t n_samples);
int lsd_frame_energy(lsd_handle* h, const float* pcm, int64_t n_samples, float* energy_out, void* stream);
int lsd_vad_mask(lsd_handle* h, const float* energy, int n_frames, float threshold, uint8_t* mask_out, void* stream);

/* ---- introspection (tests / profiling) ------------------------------------------------------- */
/* Named intermediate of the last lsd_forward on this handle: byte offset into the workspace. */
int lsd_stage_info(lsd_handle* h, const char* name, size_t* offset_bytes, int64_t* numel, int* dtype);
int lsd_stage_count(lsd_handle* h);
const char* lsd_stage_name(lsd_handle* h, int i);
/* ---- host-side transport helper (no GPU work; needs no handle) -------------------------------------------------- */
/* The reference builds float windows from uint8 mouth crops as astype(float32) / 255.0 (app/preprocessing/video.py:552-556), so
 * the pixels of a window given to _run_chunked_inference (predictor.py:554-580) are exactly fl(k / 255.0f), k in 0..255.  This
 * call verifies that for all n values of `src` (by redoing the division) while writing the k's to `dst`, on `threads` host
 * threads (0 = all).  Returns 1 when every value qualified (dst complete: ship it as LSD_U8 in the same layout — the device
 * normalisation reproduces the fp32 values bit for bit), 0 when some value did not (dst undefined: ship the fp32 values),
 * LSD_ERR_ARG on null pointers. */
int lsd_host_pack_u8_exact(const float* src, uint8_t* dst, int64_t n, int threads);
/* The same in two steps, for callers that enqueue GPU work for batch k while the host threads pack batches k+1 and k+2: _begin
 * queues the job for `threads` pool threads and returns LSD_OK at once (LSD_ERR_ARG: bad arguments, or two jobs are already in
 * flight — jobs run in submission order, the threads go from one straight on to the next); _end waits for the OLDEST job in flight
 * and returns 1 / 0 like lsd_host_pack_u8_exact (0 also when none is in flight).  src and dst must stay valid in between.
 * lsd_host_pack_u8_exact returns LSD_ERR_ARG while a _begin job is in flight. */
int lsd_host_pack_u8_begin(const float* src, uint8_t* dst, int64_t n, int threads);
int lsd_host_pack_u8_end(void);
/* Duration of the pack job the last _end (or _exact) returned, first thread started .. last thread done, in milliseconds. */
double lsd_host_pack_last_ms(void);
/* The device side of a SPLIT transport: dst[i] = fl(src[i] / 255.0f) for n device bytes, bit for bit what astype(float32) / 255.0
 * (app/preprocessing/video.py:552-556) gives on the host.  A caller whose host threads pack slower than the GPU scores sends part of
 * a batch as fp32 over PCIe and the rest packed, expands the packed part next to the fp32 part and scores one fp32 batch.  Asynchronous
 * on `stream`; n and both pointers must be multiples of 16 (bytes / elements).  Returns LSD_OK or LSD_ERR_ARG / LSD_ERR_CUDA. */
int lsd_expand_u8(const uint8_t* src, float* dst, int64_t n, void* stream);

/* CUDA-graph support.  lsd_forward may be captured into a CUDA graph (cudaStreamBeginCapture on `stream`; the internal side
 * streams join the capture through events) once a plain call with the same arguments has run: the first call of a shape
 * allocates and uploads its stage programs, which is not capturable.  A captured graph bakes in device addresses owned by the
 * handle (packed weights, stage programs); lsd_state_generation() changes whenever those are invalidated (lsd_load_weights,
 * stage-program arena recycled) — re-capture when it differs from the value read at capture time. */
int64_t lsd_state_generation(lsd_handle* h);

/* Activation tensor of the last tensor-core (BF16) lsd_forward, kept in the workspace in the padded planar bf16 layout
 * (DESIGN.md §4), converted to fp32 channels-last (N, T, H_full, W_full, C) for per-stage parity tests.  Names: "x1" (stem +
 * pool), "y1".."y4" (visual_encoder.layer1..4; y1..y3 are parity-split: pass the full-resolution extent), "ya4" (+ "ya4_lo":
 * audio_encoder.layer4), "hf_f" / "hf_b" (high-frequency branch), "art_b", "artd_b" (artifact branch). */
int lsd_planar_stage_read(lsd_handle* h, const char* name, const char* name_lo_or_null, const void* workspace, float* out,
                          int64_t out_elems, int H_full, int W_full, void* stream);
/* Number of kernels this library launched on behalf of the handle since creation. */
int64_t lsd_launch_count(lsd_handle* h);
/* Roofline instrumentation (bench.py): while enabled, every launch of the dominant kernel class (the implicit-GEMM
 * convolution / linear kernel of the selected precision) is bracketed by CUDA events on the launching stream.
 * lsd_profile_get synchronises on the recorded events, returns their summed duration, the launch count and the
 * algorithmic FLOPs (2*M*N*K per launch, padding taps counted as dense), and resets the accumulators. */
int lsd_profile_enable(lsd_handle* h, int kernel_class); /* 0 off, 1 fp32 conv kernel, 2 tcgen05 kernel: 3-D conv visual encoder launches,
                                                             3 tcgen05 kernel: all other launches (audio encoder, token GEMMs, artifact branch) */
int lsd_profile_get(lsd_handle* h, double* kernel_ms, int64_t* launches, double* flops);

#ifdef __cplusplus
}
#endif
#endif /* LSD_B200_H */
