// Occluded windows for lsd_score_occlusions: row j of a batch is one (window, box) pair; its T frames are written one after
// another into a pseudo-track of nb*T frames, which the plain scoring path then reads with window starts 0, T, 2T, ...
//   out[t,y,x,:] = (t0<=t<t1 && y0<=y<y1 && x0<=x<x1) ? (src < 0 ? fill : win[src,y,x,:]) : win[t,y,x,:]
// win = frames s_i .. s_i+T-1 of the track (the un-occluded window); only those frames are read.
// The masked log-mel windows of lsd_score_audio_occlusions are built the same way, as a pseudo clip (mask_audio_windows_kernel).
#include "lsd_kernels.h"

namespace lsd {
namespace {

// Bytes of the 16-byte chunk at byte c0 of an H x W x 3 frame that belong to pixels inside [y0,y1) x [x0,x1): bit b <-> byte b.
__device__ __forceinline__ uint32_t box_byte_mask(int c0, int W, int y0, int y1, int x0, int x1) {
  const int qa = c0 / 3, qb = (c0 + 15) / 3;   // first and last pixel the chunk touches
  int y = qa / W, x = qa - y * W;
  if (qb / W < y0 || y >= y1) return 0u;       // every pixel of the chunk lies in rows outside the box
  uint32_t m = 0;
  for (int p = 3 * qa - c0; p < 16; p += 3) {  // p: first byte of the pixel, relative to the chunk (-2..15)
    if (y >= y0 && y < y1 && x >= x0 && x < x1) {
      const int lo = p < 0 ? 0 : p, hi = p + 3 > 16 ? 16 : p + 3;
      m |= ((1u << hi) - 1u) & ~((1u << lo) - 1u);
    }
    if (++x == W) { x = 0; ++y; }
  }
  return m;
}

__device__ __forceinline__ uint32_t select_bytes(uint32_t a, uint32_t b, uint32_t bits4) {   // byte q from b where bit q is set
  uint32_t sel = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q)
    if (bits4 & (1u << q)) sel |= 0xffu << (8 * q);
  return (a & ~sel) | (b & sel);
}

// One block per output frame (row j = blockIdx.x / T, frame t).  Rows r0 .. r0+nb-1 of the call are (window r / K, box r % K);
// win_starts holds the track start of windows r0 / K, r0 / K + 1, ...; boxes: K x 7 int32 (t0, t1, y0, y1, x0, x1, src).
// VEC: 16-byte loads and stores (track, out and the frame size 16-byte aligned); only chunks a box edge cuts go byte by byte.
template <bool VEC>
__global__ void __launch_bounds__(256) occlude_windows_kernel(const uint8_t* __restrict__ track, const int32_t* __restrict__ win_starts,
                                                              const int32_t* __restrict__ boxes, int K, int r0, int T, int H, int W,
                                                              uint32_t fill, uint8_t* __restrict__ out) {
  const int j = blockIdx.x / T, t = blockIdx.x - j * T;
  const int r = r0 + j;
  const int wi = r / K, k = r - wi * K;
  const int32_t* bx = boxes + 7 * k;
  const int t0 = bx[0], t1 = bx[1], y0 = bx[2], y1 = bx[3], x0 = bx[4], x1 = bx[5], src = bx[6];
  const int64_t fb = (int64_t)H * W * 3;
  const uint8_t* win = track + (int64_t)win_starts[wi - r0 / K] * fb;
  const uint8_t* cur = win + t * fb;
  uint8_t* dst = out + (int64_t)blockIdx.x * fb;
  const bool in_t = t0 <= t && t < t1 && y0 < y1 && x0 < x1;            // this frame has pixels inside the box
  const uint8_t* rep = in_t && src >= 0 ? win + (int64_t)src * fb : nullptr;
  const bool whole = in_t && y0 == 0 && y1 == H && x0 == 0 && x1 == W;
  if (VEC) {
    const int n16 = (int)(fb / 16);
    const uint32_t f4 = fill * 0x01010101u;
    const uint4 fv = make_uint4(f4, f4, f4, f4);
    for (int c = threadIdx.x; c < n16; c += blockDim.x) {
      const uint32_t m = whole ? 0xffffu : (in_t ? box_byte_mask(c * 16, W, y0, y1, x0, x1) : 0u);
      uint4 v;
      if (m == 0xffffu) {
        v = rep ? reinterpret_cast<const uint4*>(rep)[c] : fv;
      } else {
        v = reinterpret_cast<const uint4*>(cur)[c];
        if (m) {
          const uint4 b = rep ? reinterpret_cast<const uint4*>(rep)[c] : fv;
          v.x = select_bytes(v.x, b.x, m & 15u);
          v.y = select_bytes(v.y, b.y, (m >> 4) & 15u);
          v.z = select_bytes(v.z, b.z, (m >> 8) & 15u);
          v.w = select_bytes(v.w, b.w, (m >> 12) & 15u);
        }
      }
      reinterpret_cast<uint4*>(dst)[c] = v;
    }
  } else {
    const int n = (int)fb;
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const int q = e / 3, y = q / W, x = q - y * W;
      const bool inside = in_t && y >= y0 && y < y1 && x >= x0 && x < x1;
      dst[e] = inside ? (rep ? rep[e] : (uint8_t)fill) : cur[e];
    }
  }
}

}  // namespace

void launch_occlude_windows(const uint8_t* track, const int32_t* win_starts, const int32_t* boxes, int K, int r0, int nb, int T,
                            int H, int W, int fill, uint8_t* out, cudaStream_t s) {
  if (nb < 1) return;
  const size_t fb = (size_t)H * W * 3;
  const bool vec = fb % 16 == 0 && reinterpret_cast<uintptr_t>(track) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
  const unsigned grid = (unsigned)nb * (unsigned)T;
  if (vec) occlude_windows_kernel<true><<<grid, 256, 0, s>>>(track, win_starts, boxes, K, r0, T, H, W, (uint32_t)fill, out);
  else occlude_windows_kernel<false><<<grid, 256, 0, s>>>(track, win_starts, boxes, K, r0, T, H, W, (uint32_t)fill, out);
  count_launch();
}

namespace {
// Masked audio windows for lsd_score_audio_occlusions: one block per row j (window r / K, box r % K, r = r0 + j) writes the row's
// (F, Ta) slice into columns [j*Ta, (j+1)*Ta) of the pseudo clip (F, cols):
//   out[f, j*Ta + c] = (c0<=c<c1 && f0<=f<f1) ? fill : mel[f, clamp(a_i + c, 0, Ta_full-1)]
// The unmasked values are gather_audio_kernel's (kernels_f32.cu) copy of the same column.  Consecutive threads take consecutive
// columns of one bin, so every warp stores 128 contiguous bytes.
__global__ void __launch_bounds__(256) mask_audio_windows_kernel(const float* __restrict__ mel, int F, int Ta_full,
                                                                 const int32_t* __restrict__ a_starts, const int4* __restrict__ boxes,
                                                                 int K, int r0, int Ta, float fill, int64_t cols, float* __restrict__ out) {
  const int j = blockIdx.x, r = r0 + j;
  const int wi = r / K;
  const int4 b = boxes[r - wi * K];   // (c0, c1, f0, f1)
  const int a = a_starts[wi - r0 / K];
  float* dst = out + (int64_t)j * Ta;
  const int n = F * Ta;
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const int f = e / Ta, c = e - f * Ta;
    float v;
    if (c >= b.x && c < b.y && f >= b.z && f < b.w) {
      v = fill;
    } else {
      int col = a + c;
      col = col >= Ta_full ? Ta_full - 1 : col;
      col = col < 0 ? 0 : col;
      v = mel[(int64_t)f * Ta_full + col];
    }
    dst[(int64_t)f * cols + c] = v;
  }
}

// Audio slices of lsd_score_audio_clips, built like mask_audio_windows_kernel with a clip per variant instead of a box: row j
// (window r / K, variant r % K, r = r0 + j) gets
//   out[f, j*Ta + c] = mels[k][f, clamp(a_i + c, 0, Ta_full-1)]
// mels: (K, F, Ta_full), the copy gather_audio_kernel makes of mels[k].
__global__ void __launch_bounds__(256) gather_audio_variants_kernel(const float* __restrict__ mels, int F, int Ta_full,
                                                                    const int32_t* __restrict__ a_starts, int K, int r0, int Ta,
                                                                    int64_t cols, float* __restrict__ out) {
  const int j = blockIdx.x, r = r0 + j;
  const int wi = r / K;
  const float* mel = mels + (int64_t)(r - wi * K) * F * Ta_full;
  const int a = a_starts[wi - r0 / K];
  float* dst = out + (int64_t)j * Ta;
  const int n = F * Ta;
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const int f = e / Ta, c = e - f * Ta;
    int col = a + c;
    col = col >= Ta_full ? Ta_full - 1 : col;
    col = col < 0 ? 0 : col;
    dst[(int64_t)f * cols + c] = mel[(int64_t)f * Ta_full + col];
  }
}

}  // namespace

void launch_gather_audio_variants(const float* mels, int F, int Ta_full, const int32_t* a_starts, int K, int r0, int nb, int Ta,
                                  float* out, cudaStream_t s) {
  if (nb < 1) return;
  gather_audio_variants_kernel<<<(unsigned)nb, 256, 0, s>>>(mels, F, Ta_full, a_starts, K, r0, Ta, (int64_t)nb * Ta, out);
  count_launch();
}

void launch_mask_audio_windows(const float* mel_full, int F, int Ta_full, const int32_t* a_starts, const int32_t* boxes, int K,
                               int r0, int nb, int Ta, float fill, float* out, cudaStream_t s) {
  if (nb < 1) return;
  mask_audio_windows_kernel<<<(unsigned)nb, 256, 0, s>>>(mel_full, F, Ta_full, a_starts, reinterpret_cast<const int4*>(boxes), K, r0,
                                                         Ta, fill, (int64_t)nb * Ta, out);
  count_launch();
}

}  // namespace lsd
