// Down- and re-upscaled windows for lsd_score_resizes: row j of a batch is one (window, variant) pair; frame t of the window is
// shrunk to the variant's face size and scaled back to the crop size, and written into a pseudo-track of nb*T frames, which the
// plain scoring path then reads with window starts 0, T, 2T, ... (the layout of warp_windows_kernel / jpeg_windows_kernel).  The
// frame is
//   cv2.resize(cv2.resize(frame, (w, h), interpolation=INTER_AREA), (W, H), interpolation=INTER_LINEAR)
// bit for bit: once the host has tabulated both passes' indices and weights (resize_tables below), INTER_AREA is integer or
// float32 arithmetic in a fixed order and INTER_LINEAR is 11-bit fixed point (tests/test_resize.py checks a numpy restatement
// of both against cv2 and this kernel against that).
#include "lsd_kernels.h"
#include "umma.cuh"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>

namespace lsd {
namespace {

constexpr int RESIZE_THREADS = 256;
constexpr int RESIZE_PIX = 16;                     // up pass: pixels per thread and step, 48 bytes, three 16-byte stores
constexpr int RESIZE_SMEM_MAX = 227 * 1024;        // opt-in shared memory per block on sm_100

// modes of a variant's down pass
constexpr int RS_COPY = 0, RS_AREA2 = 1, RS_AREA_INT = 2, RS_AREA = 3;

// Offsets (int32) into one variant's table, RESIZE tables of an H x W crop:
//   [mode, h, w, kx, ky, 1/(kx*ky) as float bits, 0, 0]
//   INTER_AREA taps along x: first tap of output column d at xs[d] (w + 1 used), source column xi[], float weight xw[] (<= 2W taps);
//   the same along y: ys[] (h + 1 used), yi[], yw[] (<= 2H taps)
//   INTER_LINEAR along x: source columns lx0[W], lx1[W] and coefficients la0[W], la1[W]; along y: ly0[H], ly1[H], lb0[H], lb1[H]
struct ResizeTab {
  int xs, xi, xw, ys, yi, yw, lx, ly, ints;
  __host__ __device__ ResizeTab(int H, int W) {
    xs = 8; xi = xs + W + 1; xw = xi + 2 * W;
    ys = xw + 2 * W; yi = ys + H + 1; yw = yi + 2 * H;
    lx = yw + 2 * H; ly = lx + 4 * W; ints = ly + 4 * H;
  }
};

__host__ __device__ inline int resize_frame_off(int H, int W) { return 16 + ((ResizeTab(H, W).ints * 4 + 15) & ~15); }
__host__ __device__ inline int resize_small_off(int H, int W) { return resize_frame_off(H, W) + ((H * W * 3 + 15) & ~15); }
size_t resize_smem_bytes(int H, int W) { return (size_t)resize_small_off(H, W) + (size_t)H * W * 3; }

// One block per output frame (row j = blockIdx.x / T, frame t).  Rows r0 .. r0+nb-1 of the call are (window r / K, variant r % K);
// win_starts holds the track start of windows r0 / K, r0 / K + 1, ...; tabs holds ResizeTab(H, W).ints int32 per variant.
// The source frame is staged in shared memory (one cp.async.bulk when VEC, coalesced byte loads otherwise); the down pass writes the
// h x w frame to shared memory, one thread per pixel; the up pass computes 16 output pixels per thread from it.
// VEC: track, out and the frame size are 16-byte aligned: bulk staging and 16-byte stores.
template <bool VEC>
__global__ void __launch_bounds__(RESIZE_THREADS) resize_windows_kernel(const uint8_t* __restrict__ track, const int32_t* __restrict__ win_starts,
                                                                        const int32_t* __restrict__ tabs, int K, int r0, int T, int H, int W,
                                                                        uint8_t* __restrict__ out) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int j = blockIdx.x / T, t = blockIdx.x - j * T;
  const int r = r0 + j;
  const int wi = r / K, k = r - wi * K;
  const int fb = H * W * 3;
  const uint8_t* src = track + ((int64_t)win_starts[wi - r0 / K] + t) * fb;
  uint8_t* dst = out + (int64_t)blockIdx.x * fb;
  const ResizeTab L(H, W);
  const int32_t* tg = tabs + (int64_t)k * L.ints;
  if (tg[0] == RS_COPY) {
    if (VEC) {
      for (int c = threadIdx.x; c < fb / 16; c += RESIZE_THREADS)
        reinterpret_cast<uint4*>(dst)[c] = reinterpret_cast<const uint4*>(src)[c];
    } else {
      for (int e = threadIdx.x; e < fb; e += RESIZE_THREADS) dst[e] = src[e];
    }
    return;
  }
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
  int32_t* tab = reinterpret_cast<int32_t*>(smem + 16);
  uint8_t* frame = smem + resize_frame_off(H, W);
  uint8_t* small = smem + resize_small_off(H, W);
  if (VEC && threadIdx.x == 0) {
    umma::mbar_init(bar, 1);
    umma::fence_barrier_init();
    umma::mbar_arrive_expect_tx(bar, (uint32_t)fb);
    umma::bulk_g2s(frame, src, (uint32_t)fb, bar);
  }
  if (!VEC)
    for (int e = threadIdx.x; e < fb; e += RESIZE_THREADS) frame[e] = src[e];
  for (int e = threadIdx.x; e < L.ints; e += RESIZE_THREADS) tab[e] = tg[e];
  __syncthreads();
  if (VEC) umma::mbar_wait(bar, 0);
  const int mode = tab[0], h = tab[1], w = tab[2];
  // down pass: INTER_AREA to h x w
  if (mode == RS_AREA) {
    const int32_t *xs = tab + L.xs, *xi = tab + L.xi, *xw = tab + L.xw, *ys = tab + L.ys, *yi = tab + L.yi, *yw = tab + L.yw;
    for (int q = threadIdx.x; q < h * w; q += RESIZE_THREADS) {
      const int dy = q / w, dx = q - dy * w;
      float acc[3] = {0.f, 0.f, 0.f};
      for (int a = ys[dy]; a < ys[dy + 1]; ++a) {
        const uint8_t* row = frame + yi[a] * W * 3;
        float rs[3] = {0.f, 0.f, 0.f};
        for (int b = xs[dx]; b < xs[dx + 1]; ++b) {
          const uint8_t* p = row + xi[b] * 3;
          const float wx = __int_as_float(xw[b]);
#pragma unroll
          for (int c = 0; c < 3; ++c) rs[c] = __fadd_rn(rs[c], __fmul_rn((float)p[c], wx));
        }
        const float wy = __int_as_float(yw[a]);
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[c] = __fadd_rn(acc[c], __fmul_rn(rs[c], wy));
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) small[q * 3 + c] = (uint8_t)min(max(__float2int_rn(acc[c]), 0), 255);
    }
  } else {
    const int kx = tab[3], ky = tab[4];
    const float inv = __int_as_float(tab[5]);
    for (int q = threadIdx.x; q < h * w; q += RESIZE_THREADS) {
      const int dy = q / w, dx = q - dy * w;
      int sum[3] = {0, 0, 0};
      for (int a = 0; a < ky; ++a) {
        const uint8_t* p = frame + ((dy * ky + a) * W + dx * kx) * 3;
        for (int b = 0; b < 3 * kx; b += 3) {
#pragma unroll
          for (int c = 0; c < 3; ++c) sum[c] += p[b + c];
        }
      }
#pragma unroll
      for (int c = 0; c < 3; ++c)
        small[q * 3 + c] = (uint8_t)(mode == RS_AREA2 ? (sum[c] + 2) >> 2 : min(__float2int_rn(__fmul_rn((float)sum[c], inv)), 255));
    }
  }
  __syncthreads();
  // up pass: INTER_LINEAR to H x W, 16 pixels (48 bytes) per thread and step
  const int32_t *lx0 = tab + L.lx, *lx1 = lx0 + W, *la0 = lx1 + W, *la1 = la0 + W;
  const int32_t *ly0 = tab + L.ly, *ly1 = ly0 + H, *lb0 = ly1 + H, *lb1 = lb0 + H;
  const int npix = H * W;
  for (int p0 = RESIZE_PIX * threadIdx.x; p0 < npix; p0 += RESIZE_PIX * RESIZE_THREADS) {
    const int n = npix - p0 < RESIZE_PIX ? npix - p0 : RESIZE_PIX;
    int y = p0 / W, x = p0 - y * W;
    uint32_t v[3 * RESIZE_PIX / 4] = {};
#pragma unroll
    for (int q = 0; q < RESIZE_PIX; ++q) {
      if (q < n) {
        const uint8_t* r0p = small + ly0[y] * w * 3;
        const uint8_t* r1p = small + ly1[y] * w * 3;
        const int xa = lx0[x] * 3, xb = lx1[x] * 3, a0 = la0[x], a1 = la1[x], b0 = lb0[y], b1 = lb1[y];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int R0 = a0 * r0p[xa + c] + a1 * r0p[xb + c];
          const int R1 = a0 * r1p[xa + c] + a1 * r1p[xb + c];
          // cv2's VResizeLinearVec_32s8u: the weights are >= 0 and sum to 2048, so the result lies in 0..255
          const uint32_t o = (uint32_t)((((b0 * (R0 >> 4)) >> 16) + ((b1 * (R1 >> 4)) >> 16) + 2) >> 2);
          v[(3 * q + c) >> 2] |= o << (8 * ((3 * q + c) & 3));
        }
      }
      if (++x == W) { x = 0; ++y; }
    }
    uint8_t* d = dst + 3 * p0;
    if (VEC && n == RESIZE_PIX) {
      uint4* d4 = reinterpret_cast<uint4*>(d);
      d4[0] = make_uint4(v[0], v[1], v[2], v[3]);
      d4[1] = make_uint4(v[4], v[5], v[6], v[7]);
      d4[2] = make_uint4(v[8], v[9], v[10], v[11]);
    } else {
#pragma unroll
      for (int b = 0; b < 3 * RESIZE_PIX; ++b)
        if (b < 3 * n) d[b] = (uint8_t)(v[b >> 2] >> (8 * (b & 3)));
    }
  }
}

int float_bits(float f) {
  int i;
  memcpy(&i, &f, sizeof i);
  return i;
}

double inv_ratio(int src, int dst) { return 1.0 / ((double)dst / src); }

// INTER_AREA's generic taps along one axis, as computeResizeAreaTab builds them: output d reads sources si[start[d] .. start[d+1])
// with float weights; at most 2 * src taps (a source index overlaps at most two cells of width >= 1)
__attribute__((optimize("fp-contract=off"))) void area_taps(int src, int dst, int32_t* start, int32_t* si, int32_t* wt) {
  const double scale = inv_ratio(src, dst);
  int n = 0;
  for (int d = 0; d < dst; ++d) {
    start[d] = n;
    const double f1 = d * scale, f2 = f1 + scale;
    const double cell = std::min(scale, src - f1);
    int s1 = (int)std::ceil(f1), s2 = (int)std::floor(f2);
    s2 = std::min(s2, src - 1);
    s1 = std::min(s1, s2);
    if (s1 - f1 > 1e-3) { si[n] = s1 - 1; wt[n++] = float_bits((float)((s1 - f1) / cell)); }
    for (int s = s1; s < s2; ++s) { si[n] = s; wt[n++] = float_bits((float)(1.0 / cell)); }
    if (f2 - s2 > 1e-3) { si[n] = s2; wt[n++] = float_bits((float)(std::min(std::min(f2 - s2, 1.0), cell) / cell)); }
  }
  start[dst] = n;
}

// INTER_LINEAR's taps along one axis: the two source indices read (clamped to 0 .. src-1) and the 11-bit coefficients.  Columns
// (clamp) clamp the position and zero the fraction at the borders; rows keep the fraction and only clamp the indices.
__attribute__((optimize("fp-contract=off"))) void linear_taps(int src, int dst, bool clamp, int32_t* i0, int32_t* i1, int32_t* c0, int32_t* c1) {
  const double scale = inv_ratio(src, dst);
  for (int d = 0; d < dst; ++d) {
    float f = (float)((d + 0.5) * scale - 0.5);
    int s = (int)std::floor(f);
    f -= (float)s;
    if (clamp && s < 0) { s = 0; f = 0.f; }
    if (clamp && s >= src - 1) { s = src - 1; f = 0.f; }
    i0[d] = std::min(std::max(s, 0), src - 1);
    i1[d] = std::min(std::max(s + 1, 0), src - 1);
    c0[d] = (int32_t)std::lrint((1.f - f) * 2048.f);
    c1[d] = (int32_t)std::lrint(f * 2048.f);
  }
}

// the integer ratio src / dst when INTER_AREA takes its integer path on this axis, else 0
int area_int_ratio(int src, int dst) {
  const double scale = inv_ratio(src, dst);
  const int k = (int)std::lrint(scale);
  return std::fabs(scale - k) < DBL_EPSILON ? k : 0;
}

}  // namespace

// the kernel keeps its tables, the source frame and the small frame in dynamic shared memory
cudaError_t resize_windows_device_init() {
  cudaError_t e = cudaSuccess;
  for (const void* f : {(const void*)resize_windows_kernel<true>, (const void*)resize_windows_kernel<false>})
    if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, RESIZE_SMEM_MAX);
  return e;
}

bool resize_extents_ok(int H, int W) {
  return H >= 1 && W >= 1 && (int64_t)H * W * 3 <= INT32_MAX / 4 && resize_smem_bytes(H, W) <= (size_t)RESIZE_SMEM_MAX;
}

size_t resize_tables_ints(int K, int H, int W) { return (size_t)K * ResizeTab(H, W).ints; }

// Tables of K face sizes hw (h, w pairs, 1 <= h <= H, 1 <= w <= W, checked by the caller) for an H x W crop, in the kernel's layout.
void resize_tables(const int32_t* hw, int K, int H, int W, int32_t* out) {
  const ResizeTab L(H, W);
  for (int k = 0; k < K; ++k) {
    int32_t* o = out + (size_t)k * L.ints;
    std::fill(o, o + L.ints, 0);
    const int h = hw[2 * k], w = hw[2 * k + 1];
    o[1] = h;
    o[2] = w;
    if (h == H && w == W) continue;                                   // RS_COPY
    const int kx = area_int_ratio(W, w), ky = area_int_ratio(H, h);
    if (kx && ky) {
      o[0] = kx == 2 && ky == 2 ? RS_AREA2 : RS_AREA_INT;
      o[3] = kx;
      o[4] = ky;
      o[5] = float_bits(1.f / (float)(kx * ky));
    } else {
      o[0] = RS_AREA;
      area_taps(W, w, o + L.xs, o + L.xi, o + L.xw);
      area_taps(H, h, o + L.ys, o + L.yi, o + L.yw);
    }
    linear_taps(w, W, true, o + L.lx, o + L.lx + W, o + L.lx + 2 * W, o + L.lx + 3 * W);
    linear_taps(h, H, false, o + L.ly, o + L.ly + H, o + L.ly + 2 * H, o + L.ly + 3 * H);
  }
}

void launch_resize_windows(const uint8_t* track, const int32_t* win_starts, const int32_t* tabs, int K, int r0, int nb, int T, int H, int W,
                           uint8_t* out, cudaStream_t s) {
  if (nb < 1) return;
  const size_t fb = (size_t)H * W * 3;
  const bool vec = fb % 16 == 0 && reinterpret_cast<uintptr_t>(track) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
  const size_t smem = resize_smem_bytes(H, W);
  const unsigned grid = (unsigned)nb * (unsigned)T;
  if (vec) resize_windows_kernel<true><<<grid, RESIZE_THREADS, smem, s>>>(track, win_starts, tabs, K, r0, T, H, W, out);
  else resize_windows_kernel<false><<<grid, RESIZE_THREADS, smem, s>>>(track, win_starts, tabs, K, r0, T, H, W, out);
  count_launch();
}

}  // namespace lsd
