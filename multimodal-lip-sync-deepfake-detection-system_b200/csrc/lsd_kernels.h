// Internal launcher declarations shared by the C-ABI layer (lsd_api.cu) and the kernel files.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace lsd {

enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_GELU = 2 };

// Generic fp32 implicit-GEMM convolution over channels-last activations (CUDA-core FFMA parity path).
// x: pixels of Cin contiguous floats, pixel stride in_ld;  logical extent (N, Ti, Hi, Wi).
// w: [kt*kh*kw][Cin][w_ld] (first Cout columns used).  y[row(m)*out_ld + c] for output position m.
// Linear layers are the 1-tap case (Ti=Hi=1, Wi=rows).
struct ConvF32 {
  const float* x; const float* w; const float* scale; const float* shift; const float* res; float* y;
  int N, Ti, Hi, Wi, Cin;
  int To, Ho, Wo, Cout;
  int kt, kh, kw, st, sh, sw, pt, ph, pw;
  int in_ld, w_ld, out_ld, res_ld;
  int act;
  // optional output row remap: row = (m / grp) * grp_stride + (m % grp) + row_off  (grp == 0: identity)
  int grp, grp_stride, row_off;
};
void launch_conv_f32(const ConvF32& p, cudaStream_t s);

// ---- layout / glue kernels (fp32 activations) --------------------------------------------------
// (N,C,T,H,W) of dtype -> (N,T,H,W,C) fp32
void launch_video_to_ndhwc(const void* src, int dtype, float* dst, int N, int C, int T, int H, int W, cudaStream_t s);
// same-layout cast to fp32 (audio (N,1,F,Ta) == (N,F,Ta,1); NDHWC video of another dtype); dst = src / div
void launch_cast_to_f32(const void* src, int dtype, float* dst, int64_t n, float div, cudaStream_t s);
// uint8 track (frames,H,W,3) + window starts -> (n,T,H,W,3) fp32 = u8/255 (video.py:552-556)
void launch_gather_windows_u8(const uint8_t* track, int n_frames, const int32_t* starts, float* dst,
                              int n, int T, int frame_elems, cudaStream_t s);
// occluded windows (occlusion.cu): rows r0 .. r0+nb-1 = (window r / K, box r % K) -> uint8 pseudo-track out (nb*T, H, W, 3);
// win_starts: track start of windows r0 / K, r0 / K + 1, ...; boxes: K x 7 int32 (t0, t1, y0, y1, x0, x1, src)
void launch_occlude_windows(const uint8_t* track, const int32_t* win_starts, const int32_t* boxes, int K, int r0, int nb, int T,
                            int H, int W, int fill, uint8_t* out, cudaStream_t s);
// masked audio windows (occlusion.cu): rows r0 .. r0+nb-1 = (window r / K, box r % K) -> fp32 pseudo clip out (F, nb*Ta), row j in
// columns [j*Ta, (j+1)*Ta); a_starts: base mel column of windows r0 / K, r0 / K + 1, ...; boxes: K x 4 int32 (c0, c1, f0, f1)
void launch_mask_audio_windows(const float* mel_full, int F, int Ta_full, const int32_t* a_starts, const int32_t* boxes, int K,
                               int r0, int nb, int Ta, float fill, float* out, cudaStream_t s);
// re-cropped windows (warp.cu): rows r0 .. r0+nb-1 = (window r / K, variant r % K) -> uint8 pseudo-track out (nb*T, H, W, 3), frame t
// warped like cv2.warpAffine(INTER_LINEAR, BORDER_REPLICATE) with the tables of (variant k, frame t); win_starts: track start of
// windows r0 / K, r0 / K + 1, ...; tabs: warp_tables of the K*T matrices, variant-major
void launch_warp_windows(const uint8_t* track, const int32_t* win_starts, const int32_t* tabs, int K, int r0, int nb, int T, int H, int W,
                         uint8_t* out, cudaStream_t s);
size_t warp_tables_ints(int K, int T, int H, int W);
int warp_tables(const double* m, int n, int H, int W, int32_t* out, int* bad);
cudaError_t warp_windows_device_init();
bool warp_extents_ok(int H, int W);
// mel_full (F, Ta_full) + per-window a_start -> (n, F, Ta) with repeat-last-column padding (predictor.py:525-552)
void launch_gather_audio(const float* mel_full, int F, int Ta_full, const int32_t* a_starts, float* dst,
                         int n, int Ta, cudaStream_t s);
// channels-last 3x3 / stride 2 / pad 1 max-pool over (H,W) of `frames` frames
void launch_maxpool3x3s2(const float* x, float* y, int frames, int Hi, int Wi, int C, cudaStream_t s);
// mean over the middle axis: x[A][R][Bc] -> y[a*out_ld + b]
void launch_mean_mid(const float* x, float* y, int A, int R, int Bc, int out_ld, cudaStream_t s);
// temporal difference x[:,1:] - x[:,:-1] over (N, T, S) -> (N, T-1, S)
void launch_delta_t(const float* x, float* y, int N, int T, int64_t S, cudaStream_t s);
// F.interpolate(mode=linear, align_corners=False) over tokens (N, Tin, D) -> (N, Tout, D)
void launch_lerp_tokens(const float* x, float* y, int N, int Tin, int Tout, int D, cudaStream_t s);
// y[n][0] = cls  (rows 1.. are written by the producing GEMM through the row remap)
void launch_set_cls(const float* cls, float* y, int N, int tokens, int D, cudaStream_t s);
// strided row copy: dst[r*dst_ld + c] = src[r*src_ld + c], c < width
void launch_copy_rows(const float* src, int64_t src_ld, float* dst, int64_t dst_ld, int rows, int width, cudaStream_t s);
// LayerNorm over the last axis, eps 1e-5
void launch_layernorm(const float* x, int64_t x_ld, const float* g, const float* b, float* y, int64_t y_ld, int rows, int D, cudaStream_t s);
// softmax(QK^T/sqrt(32))V, heads of 32 channels; q rows (N*Tq) with stride q_ld etc.
void launch_mha_core(const float* q, int q_ld, const float* k, int k_ld, const float* v, int v_ld,
                     float* o, int o_ld, int N, int Tq, int Tk, int heads, cudaStream_t s);
// g = sigmoid(h . w2 + b2);  out = g * v + (1-g) * a   (fusion_module.py:84-86); D channels
void launch_gate_blend(const float* h, const float* w2, const float* b2, const float* v, int v_ld,
                       const float* a, int a_ld, float* out, int rows, int D, cudaStream_t s);
// logit = LN(x) . w + b  (classifier.py:17-19)
void launch_ln_dot(const float* x, const float* g, const float* b, const float* w, const float* bias,
                   float* out, int rows, int D, cudaStream_t s);
void launch_fill_zero(float* x, int64_t n, cudaStream_t s);

// ---- log-mel (logmel.cu) -------------------------------------------------------------------------
// One clip: pcm (n_samples) -> mel power (80, frames) + atomic max into clip_max[0].
void launch_logmel_power(const float* pcm, int64_t n_samples, int frames, const float* hann, const float* twid_cos,
                         const float* twid_sin, const float* melw, const int* mel_lo, const int* mel_cnt,
                         float* mel_power, float* clip_max, cudaStream_t s);
void launch_logmel_db(float* mel, int64_t n, const float* clip_max, cudaStream_t s);
// batched FFT version (product path): clip table in device memory, one launch for all clips + one dB pass
struct LmClip { long long pcm_off, n_samples, mel_off; int frames, block0; };
size_t logmel_fft_smem_bytes();
int logmel_frames_per_block();
void init_logmel_fft_constants();
void launch_logmel_fft(const float* pcm, const LmClip* clips, int n_clips, int total_blocks, int max_frames, const float* hann,
                       const float2* w400, const float* melw, const int* mel_lo, const int* mel_cnt, float* mel_out, float* clip_max,
                       cudaStream_t s);


int64_t kernel_launches();   // process-wide count of kernels launched by this library
void count_launch(int n = 1);

// ---- speaking alignment / mouth motion (speech_stats.cu) ---------------------------------------------------
void launch_track_motion(const void* video, int layout, int n_frames, int H, int W, float* motion_full, float* motion_low, cudaStream_t s);
int speech_stats_max();
void launch_speech_stats(const float* motion_full, const float* motion_low, const int32_t* v_starts, const int32_t* a_starts, int n_windows,
                         int T, const float* mel, int F, int Ta_full, int Ta, float* score, float* mouth_motion, float* audio_energy,
                         cudaStream_t s);

void launch_frame_energy(const float* pcm, long long n, int n_frames, float* energy, cudaStream_t s);
void launch_vad_mask(const float* energy, int n_frames, float threshold, uint8_t* mask, cudaStream_t s);

}  // namespace lsd
