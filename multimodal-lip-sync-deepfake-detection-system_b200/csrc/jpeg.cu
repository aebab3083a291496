// JPEG round-tripped windows for lsd_score_jpeg: row j of a batch is one (window, variant) pair; frame t of the window goes through
// the variant's baseline JPEG encode + decode and is written into a pseudo-track of nb*T frames, which the plain scoring path then
// reads with window starts 0, T, 2T, ... (the layout of occlude_windows_kernel / warp_windows_kernel).  The round trip is
// cv2.imdecode(cv2.imencode('.jpg', frame, quality, sampling)) bit for bit (libjpeg-turbo, JDCT_ISLOW): entropy coding is
// lossless, so it is integer arithmetic from pixels to pixels (tests/test_jpeg.py checks a numpy restatement against cv2 and
// this kernel against that).
#include "lsd_kernels.h"
#include "../../include/lsd_b200.h"

namespace lsd {
namespace {

constexpr int JPEG_THREADS = 256;
constexpr int JPEG_SMEM_MAX = 227 * 1024;   // opt-in shared memory per block on sm_100
// int32 per 8x8 block in shared memory: 64 samples and 8 of padding, so the column threads of the four blocks a warp covers fall
// on distinct banks (block b starts at bank 8b mod 32), and a row is 32-byte aligned for two 16-byte accesses
constexpr int BLK = 72;

// jfdctint / jidctint constants (CONST_BITS = 13, PASS1_BITS = 2)
constexpr int CB = 13, P1 = 2;
constexpr int F0298 = 2446, F0390 = 3196, F0541 = 4433, F0765 = 6270, F0899 = 7373, F1175 = 9633;
constexpr int F1501 = 12299, F1847 = 15137, F1961 = 16069, F2053 = 16819, F2562 = 20995, F3072 = 25172;

__device__ __forceinline__ int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

// jfdctint along 8 samples: PASS 0 is the row pass, 1 the column pass
template <int PASS>
__device__ __forceinline__ void fdct8(int* d) {
  int t0 = d[0] + d[7], t7 = d[0] - d[7], t1 = d[1] + d[6], t6 = d[1] - d[6];
  int t2 = d[2] + d[5], t5 = d[2] - d[5], t3 = d[3] + d[4], t4 = d[3] - d[4];
  const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
  constexpr int sh = PASS == 0 ? CB - P1 : CB + P1;
  if (PASS == 0) {
    d[0] = (t10 + t11) << P1;
    d[4] = (t10 - t11) << P1;
  } else {
    d[0] = descale(t10 + t11, P1);
    d[4] = descale(t10 - t11, P1);
  }
  int z1 = (t12 + t13) * F0541;
  d[2] = descale(z1 + t13 * F0765, sh);
  d[6] = descale(z1 - t12 * F1847, sh);
  z1 = t4 + t7;
  int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7;
  const int z5 = (z3 + z4) * F1175;
  t4 *= F0298; t5 *= F2053; t6 *= F3072; t7 *= F1501;
  z1 *= -F0899; z2 *= -F2562;
  z3 = z3 * -F1961 + z5; z4 = z4 * -F0390 + z5;
  d[7] = descale(t4 + z1 + z3, sh);
  d[5] = descale(t5 + z2 + z4, sh);
  d[3] = descale(t6 + z2 + z3, sh);
  d[1] = descale(t7 + z1 + z4, sh);
}

// jidctint along 8 coefficients: PASS 0 is the column pass, 1 the row pass (before the range limit)
template <int PASS>
__device__ __forceinline__ void idct8(int* c) {
  int z1 = (c[2] + c[6]) * F0541;
  const int t2 = z1 - c[6] * F1847, t3 = z1 + c[2] * F0765;
  const int t0 = (c[0] + c[4]) << CB, t1 = (c[0] - c[4]) << CB;
  const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
  int a0 = c[7], a1 = c[5], a2 = c[3], a3 = c[1];
  z1 = a0 + a3;
  int z2 = a1 + a2, z3 = a0 + a2, z4 = a1 + a3;
  const int z5 = (z3 + z4) * F1175;
  a0 *= F0298; a1 *= F2053; a2 *= F3072; a3 *= F1501;
  z1 *= -F0899; z2 *= -F2562;
  z3 = z3 * -F1961 + z5; z4 = z4 * -F0390 + z5;
  a0 += z1 + z3; a1 += z2 + z4; a2 += z2 + z3; a3 += z1 + z4;
  constexpr int sh = PASS == 1 ? CB + P1 + 3 : CB - P1;
  c[0] = descale(t10 + a3, sh); c[7] = descale(t10 - a3, sh);
  c[1] = descale(t11 + a2, sh); c[6] = descale(t11 - a2, sh);
  c[2] = descale(t12 + a1, sh); c[5] = descale(t12 - a1, sh);
  c[3] = descale(t13 + a0, sh); c[4] = descale(t13 - a0, sh);
}

// jidctint's range limit of a descaled output centred on 0 -> sample 0..255
__device__ __forceinline__ int range_limit(int x) {
  const int m = x & 1023;
  return m < 128 ? m + 128 : (m < 512 ? 255 : (m < 896 ? 0 : m - 896));
}

__device__ __forceinline__ int ycc_y(int r, int g, int b) { return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16; }
__device__ __forceinline__ int ycc_cb(int r, int g, int b) { return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16; }
__device__ __forceinline__ int ycc_cr(int r, int g, int b) { return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16; }
__device__ __forceinline__ int clamp255(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }

// sample (y, x) of a block-major plane bw blocks wide
__device__ __forceinline__ int at(int bw, int y, int x) { return ((y >> 3) * bw + (x >> 3)) * BLK + (y & 7) * 8 + (x & 7); }

// One block per output frame (row j = blockIdx.x / T, frame t).  Rows r0 .. r0+nb-1 of the call are (window r / K, variant r % K);
// win_starts holds the track start of windows r0 / K, r0 / K + 1, ...; tabs holds JPEG_TAB_INTS int32 per variant (jpeg_tables).
// The frame's Y, Cb and Cr planes live in shared memory as int32, block-major; every 1-D DCT pass runs one thread per 8-sample
// line, and the forward column pass, quantisation, dequantisation and the inverse column pass share one thread per column.
// BGR: byte 0 of a pixel is blue (else red).  VEC: track, out and the frame size are 16-byte aligned: 16-byte loads and stores.
template <bool VEC>
__global__ void __launch_bounds__(JPEG_THREADS) jpeg_windows_kernel(const uint8_t* __restrict__ track, const int32_t* __restrict__ win_starts,
                                                                    const int32_t* __restrict__ tabs, int K, int r0, int T, int H, int W,
                                                                    int bgr, uint8_t* __restrict__ out) {
  extern __shared__ __align__(16) int32_t sp[];
  const int j = blockIdx.x / T, t = blockIdx.x - j * T;
  const int r = r0 + j;
  const int wi = r / K, k = r - wi * K;
  const int fb = H * W * 3;
  const uint8_t* src = track + ((int64_t)win_starts[wi - r0 / K] + t) * fb;
  uint8_t* dst = out + (int64_t)blockIdx.x * fb;
  const int32_t* tab = tabs + (int64_t)k * JPEG_TAB_INTS;
  const int sampling = tab[0];
  if (sampling == LSD_JPEG_NONE) {
    if (VEC) {
      for (int c = threadIdx.x; c < fb / 16; c += JPEG_THREADS)
        reinterpret_cast<uint4*>(dst)[c] = reinterpret_cast<const uint4*>(src)[c];
    } else {
      for (int e = threadIdx.x; e < fb; e += JPEG_THREADS) dst[e] = src[e];
    }
    return;
  }
  const bool sub = sampling == LSD_JPEG_420;
  const int ci = bgr ? 2 : 0, bi = bgr ? 0 : 2;      // byte offsets of red and blue in a pixel
  const int bwY = W >> 3, nbY = (H >> 3) * bwY;
  const int Hc = sub ? H >> 1 : H, Wc = sub ? W >> 1 : W, bwC = Wc >> 3, nbC = (Hc >> 3) * bwC;
  int32_t* Yp = sp;
  int32_t* Cbp = sp + nbY * BLK;
  int32_t* Crp = Cbp + nbC * BLK;
  // colour conversion (and 4:2:0 downsampling) into level-shifted planes; one thread per chroma sample
  for (int q = threadIdx.x; q < Hc * Wc; q += JPEG_THREADS) {
    const int cy = q / Wc, cx = q - cy * Wc;
    if (sub) {
      int scb = 0, scr = 0;
#pragma unroll
      for (int d = 0; d < 4; ++d) {
        const int y = 2 * cy + (d >> 1), x = 2 * cx + (d & 1);
        const uint8_t* p = src + (y * W + x) * 3;
        const int R = p[ci], G = p[1], B = p[bi];
        Yp[at(bwY, y, x)] = ycc_y(R, G, B) - 128;
        scb += ycc_cb(R, G, B);
        scr += ycc_cr(R, G, B);
      }
      const int bias = 1 + (cx & 1);
      Cbp[at(bwC, cy, cx)] = ((scb + bias) >> 2) - 128;
      Crp[at(bwC, cy, cx)] = ((scr + bias) >> 2) - 128;
    } else {
      const uint8_t* p = src + q * 3;
      const int R = p[ci], G = p[1], B = p[bi];
      const int o = at(bwY, cy, cx);
      Yp[o] = ycc_y(R, G, B) - 128;
      Cbp[o] = ycc_cb(R, G, B) - 128;
      Crp[o] = ycc_cr(R, G, B) - 128;
    }
  }
  __syncthreads();
  const int lines = (nbY + 2 * nbC) * 8;
  // forward DCT, row pass
  for (int l = threadIdx.x; l < lines; l += JPEG_THREADS) {
    int4* p = reinterpret_cast<int4*>(sp + (l >> 3) * BLK + (l & 7) * 8);
    int4 a = p[0], b = p[1];
    int d[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    fdct8<0>(d);
    p[0] = make_int4(d[0], d[1], d[2], d[3]);
    p[1] = make_int4(d[4], d[5], d[6], d[7]);
  }
  __syncthreads();
  // forward DCT column pass, quantisation (qc = sign(c) * ((|c| + d/2) / d), d = 8 * qtab, the division by a host-built
  // reciprocal: exact while |c| * d < 2^32), dequantisation, inverse DCT column pass
  for (int l = threadIdx.x; l < lines; l += JPEG_THREADS) {
    const int b = l >> 3, c = l & 7;
    int32_t* p = sp + b * BLK + c;
    const int32_t* qt = tab + (b < nbY ? JPEG_TAB_LUMA : JPEG_TAB_CHROMA);
    int d[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = p[8 * i];
    fdct8<1>(d);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int q = qt[8 * i + c];
      const uint32_t mul = (uint32_t)qt[64 + 8 * i + c];
      const int m = (int)__umulhi((uint32_t)(abs(d[i]) + 4 * q), mul);
      d[i] = (d[i] < 0 ? -m : m) * q;
    }
    idct8<0>(d);
#pragma unroll
    for (int i = 0; i < 8; ++i) p[8 * i] = d[i];
  }
  __syncthreads();
  // inverse DCT row pass and range limit: samples 0..255
  for (int l = threadIdx.x; l < lines; l += JPEG_THREADS) {
    int4* p = reinterpret_cast<int4*>(sp + (l >> 3) * BLK + (l & 7) * 8);
    int4 a = p[0], b = p[1];
    int d[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    idct8<1>(d);
    p[0] = make_int4(range_limit(d[0]), range_limit(d[1]), range_limit(d[2]), range_limit(d[3]));
    p[1] = make_int4(range_limit(d[4]), range_limit(d[5]), range_limit(d[6]), range_limit(d[7]));
  }
  __syncthreads();
  // 4:2:0 fancy upsampling, YCbCr -> RGB, 16 pixels (48 bytes) per thread and step
  const int npix = H * W;
  for (int p0 = 16 * threadIdx.x; p0 < npix; p0 += 16 * JPEG_THREADS) {
    int y = p0 / W, x = p0 - y * W;
    uint32_t v[12] = {};
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int Y = Yp[at(bwY, y, x)];
      int cb, cr;
      if (sub) {
        // h2v2_fancy_upsample: the nearer chroma row weighs 3, the farther (above for an upper output row, below for a lower
        // one, edges replicated) 1; then 3:1 across columns with rounding 8 / 7 for even / odd outputs
        const int cy = y >> 1, cx = x >> 1;
        const int fy = (y & 1) ? min(cy + 1, Hc - 1) : max(cy - 1, 0);
        const bool odd = x & 1;
        const int nx = odd ? cx + 1 : cx - 1;
        const bool edge = nx < 0 || nx >= Wc;
        const int cs0 = 3 * Cbp[at(bwC, cy, cx)] + Cbp[at(bwC, fy, cx)];
        const int cr0 = 3 * Crp[at(bwC, cy, cx)] + Crp[at(bwC, fy, cx)];
        const int cs1 = edge ? cs0 : 3 * Cbp[at(bwC, cy, nx)] + Cbp[at(bwC, fy, nx)];
        const int cr1 = edge ? cr0 : 3 * Crp[at(bwC, cy, nx)] + Crp[at(bwC, fy, nx)];
        const int rnd = odd ? 7 : 8;
        cb = (3 * cs0 + cs1 + rnd) >> 4;
        cr = (3 * cr0 + cr1 + rnd) >> 4;
      } else {
        cb = Cbp[at(bwY, y, x)];
        cr = Crp[at(bwY, y, x)];
      }
      const int xr = cr - 128, zb = cb - 128;
      const int R = clamp255(Y + ((91881 * xr + 32768) >> 16));
      const int B = clamp255(Y + ((116130 * zb + 32768) >> 16));
      const int G = clamp255(Y + ((-22554 * zb - 46802 * xr + 32768) >> 16));
      const int c0 = bgr ? B : R, c2 = bgr ? R : B;
      v[(3 * q) >> 2] |= (uint32_t)c0 << (8 * ((3 * q) & 3));
      v[(3 * q + 1) >> 2] |= (uint32_t)G << (8 * ((3 * q + 1) & 3));
      v[(3 * q + 2) >> 2] |= (uint32_t)c2 << (8 * ((3 * q + 2) & 3));
      if (++x == W) { x = 0; ++y; }
    }
    uint8_t* d = dst + 3 * p0;
    if (VEC) {
      uint4* d4 = reinterpret_cast<uint4*>(d);
      d4[0] = make_uint4(v[0], v[1], v[2], v[3]);
      d4[1] = make_uint4(v[4], v[5], v[6], v[7]);
      d4[2] = make_uint4(v[8], v[9], v[10], v[11]);
    } else {
#pragma unroll
      for (int b = 0; b < 48; ++b) d[b] = (uint8_t)(v[b >> 2] >> (8 * (b & 3)));
    }
  }
}

}  // namespace

// the planes of a 96x96 4:4:4 frame already take 124 KB
cudaError_t jpeg_windows_device_init() {
  cudaError_t e = cudaSuccess;
  for (const void* f : {(const void*)jpeg_windows_kernel<true>, (const void*)jpeg_windows_kernel<false>})
    if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, JPEG_SMEM_MAX);
  return e;
}

size_t jpeg_smem_bytes(int H, int W, bool any444) {
  const size_t nbY = (size_t)(H / 8) * (W / 8);
  return (nbY + 2 * (any444 ? nbY : nbY / 4)) * BLK * sizeof(int32_t);
}

bool jpeg_extents_ok(int H, int W, bool any444) { return jpeg_smem_bytes(H, W, any444) <= (size_t)JPEG_SMEM_MAX; }

// qs: (quality, sampling) of K variants (lsd_jpeg).  Per variant: [sampling, quality, 6 unused | luma qtab[64] | luma reciprocal[64] | chroma qtab[64] | chroma reciprocal[64]], the
// tables in natural order.  qtab: jpeg_quality_scaling + jpeg_add_quant_table with force_baseline (IJG Annex K tables);
// reciprocal: ceil(2^32 / (8 * qtab)), so (n * reciprocal) >> 32 == n / (8 * qtab) for every n with n * 8 * qtab < 2^32.
void jpeg_tables(const int32_t* qs, int K, int32_t* out) {
  static const int luma[64] = {16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
                               14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
                               49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
  static const int chroma[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99,
                                 47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
  for (int k = 0; k < K; ++k) {
    int32_t* o = out + (size_t)k * JPEG_TAB_INTS;
    for (int e = 0; e < JPEG_TAB_INTS; ++e) o[e] = 0;
    const int quality = qs[2 * k], sampling = qs[2 * k + 1];
    o[0] = sampling;
    o[1] = quality;
    const int q = quality < 1 ? 1 : (quality > 100 ? 100 : quality);
    const long s = q < 50 ? 5000 / q : 200 - 2 * q;
    for (int c = 0; c < 2; ++c) {
      const int* base = c ? chroma : luma;
      int32_t* t = o + (c ? JPEG_TAB_CHROMA : JPEG_TAB_LUMA);
      for (int i = 0; i < 64; ++i) {
        long e = (base[i] * s + 50) / 100;
        e = e < 1 ? 1 : (e > 255 ? 255 : e);
        t[i] = (int32_t)e;
        t[64 + i] = (int32_t)(uint32_t)(((1ull << 32) + 8 * e - 1) / (8 * e));
      }
    }
  }
}

void launch_jpeg_windows(const uint8_t* track, const int32_t* win_starts, const int32_t* tabs, int K, int r0, int nb, int T, int H, int W,
                         bool any444, int bgr, uint8_t* out, cudaStream_t s) {
  if (nb < 1) return;
  const size_t fb = (size_t)H * W * 3;
  const bool vec = fb % 16 == 0 && reinterpret_cast<uintptr_t>(track) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
  const size_t smem = jpeg_smem_bytes(H, W, any444);
  const unsigned grid = (unsigned)nb * (unsigned)T;
  if (vec) jpeg_windows_kernel<true><<<grid, JPEG_THREADS, smem, s>>>(track, win_starts, tabs, K, r0, T, H, W, bgr, out);
  else jpeg_windows_kernel<false><<<grid, JPEG_THREADS, smem, s>>>(track, win_starts, tabs, K, r0, T, H, W, bgr, out);
  count_launch();
}

}  // namespace lsd
