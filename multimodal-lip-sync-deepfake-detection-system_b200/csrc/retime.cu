// Retimed windows for lsd_score_retimes: row j of a batch is one (window, variant) pair; output frame t of the window is a convex
// Q15 blend of up to four frames of the caller's track near the window, and is written into a pseudo-track of nb*T frames, which
// the plain scoring path then reads with window starts 0, T, 2T, ... (the layout of warp_windows_kernel / resize_windows_kernel).
// Tap i of (variant k, frame t) names the frame clamp(window_start + src_i, 0, n_frames - 1) with weight w_i >= 0, the weights
// summing to LSD_RETIME_ONE; every byte is
//   out = (sum_i w_i * p_i + 16384) >> 15
// exact integer arithmetic (tests/test_retime.py restates it in numpy and checks this kernel against that byte for byte).  The
// weights are convex, so the result lies in 0..255 and a single full-weight tap is an exact copy.  The host builds every table
// (held, frozen, dropped, blended frames, inference.py); the kernel has no table of its own and no floating point.
#include "lsd_kernels.h"

namespace lsd {
namespace {

constexpr int RETIME_THREADS = 256;
constexpr int RETIME_TAPS = 4;
constexpr int RETIME_ENTRY_INTS = 2 * RETIME_TAPS;   // one lsd_retime: src[4], weight[4]

// One block per output frame (row j = blockIdx.x / T, frame t).  Rows r0 .. r0+nb-1 of the call are (window r / K, variant r % K);
// win_starts holds the track start of windows r0 / K, r0 / K + 1, ...; tabs holds the K*T lsd_retime entries, (variant k, frame
// t) at k*T + t.  The taps are the same for the whole block, so they live in registers and every branch on them is uniform:
// weight-0 taps are skipped, and a single full-weight tap is a plain copy (the same bits as the blend: (32768 p + 16384) >> 15 = p).
// VEC: track, out and the frame size are 16-byte aligned: every thread loads 16 bytes of each tap frame and stores 16 bytes per step.
// Otherwise byte loads and byte stores.
template <bool VEC>
__global__ void __launch_bounds__(RETIME_THREADS) retime_windows_kernel(const uint8_t* __restrict__ track, int n_frames,
                                                                        const int32_t* __restrict__ win_starts,
                                                                        const int32_t* __restrict__ tabs, int K, int r0, int T, int H,
                                                                        int W, uint8_t* __restrict__ out) {
  const int j = blockIdx.x / T, t = blockIdx.x - j * T;
  const int r = r0 + j;
  const int wi = r / K, k = r - wi * K;
  const int64_t fb = (int64_t)H * W * 3;
  const int32_t* e = tabs + ((int64_t)k * T + t) * RETIME_ENTRY_INTS;
  const int w0 = win_starts[wi - r0 / K];
  const uint8_t* src[RETIME_TAPS];
  int wt[RETIME_TAPS];
#pragma unroll
  for (int i = 0; i < RETIME_TAPS; ++i) {
    // the host checks src and the window, and the clamp keeps a tap inside the track whatever the table holds
    const int f = min(max(w0 + e[i], 0), n_frames - 1);
    src[i] = track + f * fb;
    wt[i] = e[RETIME_TAPS + i];
  }
  uint8_t* dst = out + (int64_t)blockIdx.x * fb;
  const uint8_t* copy = wt[0] == LSD_RETIME_ONE ? src[0] : wt[1] == LSD_RETIME_ONE ? src[1]
                      : wt[2] == LSD_RETIME_ONE ? src[2] : wt[3] == LSD_RETIME_ONE ? src[3] : nullptr;
  if (VEC) {
    const int n16 = (int)(fb / 16);
    if (copy) {
      for (int c = threadIdx.x; c < n16; c += RETIME_THREADS)
        reinterpret_cast<uint4*>(dst)[c] = reinterpret_cast<const uint4*>(copy)[c];
      return;
    }
    for (int c = threadIdx.x; c < n16; c += RETIME_THREADS) {
      uint4 v[RETIME_TAPS];
#pragma unroll
      for (int i = 0; i < RETIME_TAPS; ++i)
        if (wt[i]) v[i] = reinterpret_cast<const uint4*>(src[i])[c];
      uint32_t acc[16];
#pragma unroll
      for (int b = 0; b < 16; ++b) acc[b] = 1u << 14;
#pragma unroll
      for (int i = 0; i < RETIME_TAPS; ++i) {
        if (wt[i]) {
          const uint32_t q[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
#pragma unroll
          for (int b = 0; b < 16; ++b) acc[b] += (uint32_t)wt[i] * ((q[b >> 2] >> (8 * (b & 3))) & 0xffu);
        }
      }
      uint32_t o[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int b = 0; b < 16; ++b) o[b >> 2] |= (acc[b] >> 15) << (8 * (b & 3));
      reinterpret_cast<uint4*>(dst)[c] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  } else {
    if (copy) {
      for (int64_t c = threadIdx.x; c < fb; c += RETIME_THREADS) dst[c] = copy[c];
      return;
    }
    for (int64_t c = threadIdx.x; c < fb; c += RETIME_THREADS) {
      uint32_t acc = 1u << 14;
#pragma unroll
      for (int i = 0; i < RETIME_TAPS; ++i)
        if (wt[i]) acc += (uint32_t)wt[i] * src[i][c];
      dst[c] = (uint8_t)(acc >> 15);
    }
  }
}

}  // namespace

size_t retime_tables_ints(int K, int T) { return (size_t)K * T * RETIME_ENTRY_INTS; }

void launch_retime_windows(const uint8_t* track, int n_frames, const int32_t* win_starts, const int32_t* tabs, int K, int r0, int nb,
                           int T, int H, int W, uint8_t* out, cudaStream_t s) {
  if (nb < 1) return;
  const size_t fb = (size_t)H * W * 3;
  const bool vec = fb % 16 == 0 && reinterpret_cast<uintptr_t>(track) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
  const unsigned grid = (unsigned)nb * (unsigned)T;
  if (vec) retime_windows_kernel<true><<<grid, RETIME_THREADS, 0, s>>>(track, n_frames, win_starts, tabs, K, r0, T, H, W, out);
  else retime_windows_kernel<false><<<grid, RETIME_THREADS, 0, s>>>(track, n_frames, win_starts, tabs, K, r0, T, H, W, out);
  count_launch();
}

}  // namespace lsd
