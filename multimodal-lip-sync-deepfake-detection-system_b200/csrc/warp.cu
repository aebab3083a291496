// Re-cropped windows for lsd_score_warps: row j of a batch is one (window, variant) pair; frame t of the window is warped by the
// variant's matrix for frame t and written into a pseudo-track of nb*T frames, which the plain scoring path then reads with window
// starts 0, T, 2T, ... (the layout of occlude_windows_kernel).  The warp is cv2.warpAffine(src, M, (W, H), INTER_LINEAR,
// BORDER_REPLICATE) bit for bit: once its per-row and per-column terms are tabulated on the host (warp_tables below), every pixel
// is integer arithmetic (tests/test_warps.py restates it in numpy and checks that against cv2).
#include "lsd_kernels.h"
#include "umma.cuh"

#include <cmath>
#include <cstdlib>

namespace lsd {
namespace {

constexpr int WARP_THREADS = 256;
constexpr int WARP_PIX = 16;                       // pixels per thread and step: 48 bytes, three 16-byte stores
constexpr int WARP_SMEM_MAX = 227 * 1024;          // opt-in shared memory per block on sm_100

__host__ __device__ constexpr int warp_tab_ints(int H, int W) { return 2 * (H + W); }
__host__ __device__ constexpr int warp_frame_off(int H, int W) { return 16 + ((warp_tab_ints(H, W) * 4 + 15) & ~15); }

// One block per output frame (row j = blockIdx.x / T, frame t).  Rows r0 .. r0+nb-1 of the call are (window r / K, variant r % K);
// win_starts holds the track start of windows r0 / K, r0 / K + 1, ...; tabs holds (X0[H], Y0[H], adelta[W], bdelta[W]) int32 of
// (variant k, frame t) at (k*T + t) * 2(H+W).
// SMEM: the source frame is staged in shared memory (one cp.async.bulk when VEC, coalesced byte loads otherwise); without it the
// taps are read from global memory through L1 / L2 (frames too large for shared memory).
// VEC: track, out and the frame size are 16-byte aligned: bulk staging and 16-byte stores.
template <bool SMEM, bool VEC>
__global__ void __launch_bounds__(WARP_THREADS) warp_windows_kernel(const uint8_t* __restrict__ track, const int32_t* __restrict__ win_starts,
                                                                    const int32_t* __restrict__ tabs, int K, int r0, int T, int H, int W,
                                                                    uint8_t* __restrict__ out) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int j = blockIdx.x / T, t = blockIdx.x - j * T;
  const int r = r0 + j;
  const int wi = r / K, k = r - wi * K;
  const int fb = H * W * 3;
  const uint8_t* src = track + ((int64_t)win_starts[wi - r0 / K] + t) * fb;
  uint8_t* dst = out + (int64_t)blockIdx.x * fb;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
  int32_t* tab = reinterpret_cast<int32_t*>(smem + 16);
  uint8_t* frame = smem + warp_frame_off(H, W);
  if (SMEM && VEC && threadIdx.x == 0) {
    umma::mbar_init(bar, 1);
    umma::fence_barrier_init();
    umma::mbar_arrive_expect_tx(bar, (uint32_t)fb);
    umma::bulk_g2s(frame, src, (uint32_t)fb, bar);
  }
  if (SMEM && !VEC)
    for (int e = threadIdx.x; e < fb; e += WARP_THREADS) frame[e] = src[e];
  const int nt = warp_tab_ints(H, W);
  const int32_t* tg = tabs + ((int64_t)k * T + t) * nt;
  for (int e = threadIdx.x; e < nt; e += WARP_THREADS) tab[e] = tg[e];
  __syncthreads();
  if (SMEM && VEC) umma::mbar_wait(bar, 0);
  const uint8_t* img = SMEM ? frame : src;
  const int32_t *X0 = tab, *Y0 = tab + H, *adelta = tab + 2 * H, *bdelta = tab + 2 * H + W;
  const int npix = H * W;
  for (int p0 = WARP_PIX * threadIdx.x; p0 < npix; p0 += WARP_PIX * WARP_THREADS) {
    const int n = npix - p0 < WARP_PIX ? npix - p0 : WARP_PIX;
    int y = p0 / W, x = p0 - y * W;
    uint32_t v[3 * WARP_PIX / 4] = {};             // the 48 output bytes, little-endian
#pragma unroll
    for (int q = 0; q < WARP_PIX; ++q) {
      if (q < n) {
        const int X = (X0[y] + adelta[x]) >> 5, Y = (Y0[y] + bdelta[x]) >> 5;
        const int fx = X & 31, fy = Y & 31, xi = X >> 5, yi = Y >> 5;
        const int xa = min(max(xi, 0), W - 1), xb = min(max(xi + 1, 0), W - 1);
        const int ya = min(max(yi, 0), H - 1), yb = min(max(yi + 1, 0), H - 1);
        // cv2's bilinear table entry (fy, fx): every product is exact in its float arithmetic, so it is this closed form
        const int w00 = (32 - fy) * (32 - fx) * 32, w01 = (32 - fy) * fx * 32, w10 = fy * (32 - fx) * 32, w11 = fy * fx * 32;
        const uint8_t* p00 = img + (ya * W + xa) * 3;
        const uint8_t* p01 = img + (ya * W + xb) * 3;
        const uint8_t* p10 = img + (yb * W + xa) * 3;
        const uint8_t* p11 = img + (yb * W + xb) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          // the weights are >= 0 and sum to 32768, so the result lies in 0..255 without cv2's clamp
          const uint32_t o = (uint32_t)(w00 * p00[c] + w01 * p01[c] + w10 * p10[c] + w11 * p11[c] + 16384) >> 15;
          v[(3 * q + c) >> 2] |= o << (8 * ((3 * q + c) & 3));
        }
      }
      if (++x == W) { x = 0; ++y; }
    }
    uint8_t* d = dst + 3 * p0;
    if (VEC && n == WARP_PIX) {
      uint4* d4 = reinterpret_cast<uint4*>(d);
      d4[0] = make_uint4(v[0], v[1], v[2], v[3]);
      d4[1] = make_uint4(v[4], v[5], v[6], v[7]);
      d4[2] = make_uint4(v[8], v[9], v[10], v[11]);
    } else {
#pragma unroll
      for (int b = 0; b < 3 * WARP_PIX; ++b)
        if (b < 3 * n) d[b] = (uint8_t)(v[b >> 2] >> (8 * (b & 3)));
    }
  }
}

template <bool SMEM, bool VEC>
void launch_warp(unsigned grid, size_t smem, cudaStream_t s, const uint8_t* track, const int32_t* win_starts, const int32_t* tabs, int K,
                 int r0, int T, int H, int W, uint8_t* out) {
  warp_windows_kernel<SMEM, VEC><<<grid, WARP_THREADS, smem, s>>>(track, win_starts, tabs, K, r0, T, H, W, out);
}

}  // namespace

// every variant keeps its tables in dynamic shared memory, so every variant may need more than the default 48 KB
cudaError_t warp_windows_device_init() {
  cudaError_t e = cudaSuccess;
  for (const void* f : {(const void*)warp_windows_kernel<true, true>, (const void*)warp_windows_kernel<true, false>,
                        (const void*)warp_windows_kernel<false, true>, (const void*)warp_windows_kernel<false, false>})
    if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, WARP_SMEM_MAX);
  return e;
}

// the frame's tables (and the staging barrier) must fit in shared memory: H + W up to about 29 000
bool warp_extents_ok(int H, int W) { return (int64_t)H + W <= (WARP_SMEM_MAX - 32) / 8; }

size_t warp_tables_ints(int K, int T, int H, int W) { return (size_t)K * T * warp_tab_ints(H, W); }

// Tables of cv::warpAffine for K*T forward matrices (m: 6 doubles each), in the kernel's layout; returns -1 for a matrix with a
// non-finite entry or a zero determinant, -2 for one whose inverse maps a pixel of the H x W frame to |coordinate| >= 2^15 - 1
// (cv2's int16 tap coordinates would saturate), 0 otherwise; *bad is the index of the offending matrix.  Compiled without
// floating-point contraction: a fused multiply-add changes the last bit of a product and the tables would no longer be cv2's.
__attribute__((optimize("fp-contract=off"))) int warp_tables(const double* m, int n, int H, int W, int32_t* out, int* bad) {
  const double lim = 32767.0;
  for (int i = 0; i < n; ++i) {
    const double* M = m + 6 * i;
    *bad = i;
    for (int e = 0; e < 6; ++e)
      if (!std::isfinite(M[e])) return -1;
    // cv::warpAffine inverts the forward matrix itself (WARP_INVERSE_MAP not set), in this order
    double D = M[0] * M[4] - M[1] * M[3];
    if (D == 0.0) return -1;
    D = 1.0 / D;
    const double a0 = M[4] * D, a1 = -M[1] * D, a3 = -M[3] * D, a4 = M[0] * D;
    const double a2 = -a0 * M[2] - a1 * M[5], a5 = -a3 * M[2] - a4 * M[5];
    // an affine map takes its extremes over the frame at the corners; the negated tests also catch NaN
    for (int c = 0; c < 4; ++c) {
      const double x = (c & 1) ? W - 1 : 0, y = (c & 2) ? H - 1 : 0;
      const double u = a0 * x + a1 * y + a2, v = a3 * x + a4 * y + a5;
      if (!(std::fabs(u) < lim) || !(std::fabs(v) < lim)) return -2;
    }
    int32_t* X0 = out + (size_t)i * warp_tab_ints(H, W);
    int32_t *Y0 = X0 + H, *ad = X0 + 2 * H, *bd = X0 + 2 * H + W;
    for (int x = 0; x < W; ++x) {
      ad[x] = (int32_t)std::lrint(a0 * x * 1024.0);
      bd[x] = (int32_t)std::lrint(a3 * x * 1024.0);
    }
    for (int y = 0; y < H; ++y) {
      X0[y] = (int32_t)std::lrint((a1 * y + a2) * 1024.0) + 16;
      Y0[y] = (int32_t)std::lrint((a4 * y + a5) * 1024.0) + 16;
    }
  }
  return 0;
}

void launch_warp_windows(const uint8_t* track, const int32_t* win_starts, const int32_t* tabs, int K, int r0, int nb, int T, int H, int W,
                         uint8_t* out, cudaStream_t s) {
  if (nb < 1) return;
  const size_t fb = (size_t)H * W * 3;
  const bool vec = fb % 16 == 0 && reinterpret_cast<uintptr_t>(track) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
  const size_t smem_tab = (size_t)warp_frame_off(H, W);
  const bool in_smem = smem_tab + fb <= (size_t)WARP_SMEM_MAX && getenv("LSD_WARP_L2_TAPS") == nullptr;
  const size_t smem = in_smem ? smem_tab + fb : smem_tab;
  const unsigned grid = (unsigned)nb * (unsigned)T;
  if (in_smem) {
    if (vec) launch_warp<true, true>(grid, smem, s, track, win_starts, tabs, K, r0, T, H, W, out);
    else launch_warp<true, false>(grid, smem, s, track, win_starts, tabs, K, r0, T, H, W, out);
  } else {
    if (vec) launch_warp<false, true>(grid, smem, s, track, win_starts, tabs, K, r0, T, H, W, out);
    else launch_warp<false, false>(grid, smem, s, track, win_starts, tabs, K, r0, T, H, W, out);
  }
  count_launch();
}

}  // namespace lsd
