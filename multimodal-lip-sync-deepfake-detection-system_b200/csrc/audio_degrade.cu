// Degraded copies of one PCM clip for lsd_degrade_audio: K variants, each a chain of optional stages run in a fixed order
// (reverb, noise, clip, band, mu-law), written as (K, n) fp32.  tests/test_audio_robustness.py checks every stage against a numpy restatement.
//   reverb: the first n samples of x * h, h a synthetic room impulse response built on the host (fir_reverb_kernel)
//   noise:  x + sqrt(P_x / (P_g 10^(snr/10))) g, g white Gaussian from a counter-based generator, P over the clip in fp64
//   clip:   clamp(x * fl32(10^(gain/20)), -1, 1)
//   band:   scipy.signal.resample_poly(x, 1, f) then resample_poly(., f, 1), cut to n (upfirdn_kernel, both passes)
//   mu-law: int16 = clamp(rint(x * 32768)), audioop.lin2ulaw / ulaw2lin (Sun G.711 on 14-bit values), / 32768
// Every kernel takes the variant from blockIdx.y and returns at once when the variant lacks its stage.
#include "lsd_kernels.h"
#include "../../include/lsd_b200.h"

#include <cmath>
#include <cstring>
#include <vector>

namespace lsd {
namespace {

constexpr int SR = 16000;
// FIR tiling: 256 threads x 8 consecutive outputs per CTA, taps in chunks of 2048; shared: the chunk's taps and the
// 2048 + 2048 input samples it meets, plus 4 samples of front padding for the last window load
constexpr int FIR_THREADS = 256, FIR_R = 8, FIR_TO = FIR_THREADS * FIR_R, FIR_TJ = 2048;
constexpr int POW_BLOCKS = 128;   // per-variant partial sums of the noise stage (summed in a fixed order: deterministic)

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// Draw i of (seed, stream): two 24-bit uniforms of splitmix64(key + i), Box-Muller in double.
__host__ __device__ __forceinline__ double gauss(uint64_t key, uint64_t i) {
  const uint64_t r = splitmix64(key + i);
  const double u1 = (double)((r >> 40) + 1) * 0x1p-24, u2 = (double)((r >> 16) & 0xFFFFFFu) * 0x1p-24;
  return sqrt(-2.0 * log(u1)) * cos(2.0 * 3.141592653589793 * u2);
}
__host__ __device__ __forceinline__ uint64_t stream_key(uint32_t seed, uint32_t stream) {
  return splitmix64(((uint64_t)seed << 32) | stream);
}

struct VarTab {   // the per-variant words of the device table (DEGRADE_TAB_INTS int32)
  int32_t stages, rir_len, rir_off, f;
  float gain;
  uint32_t seed;
  double snr_lin;   // 10^(snr/10)
};
static_assert(sizeof(VarTab) == DEGRADE_TAB_INTS * sizeof(int32_t), "VarTab is DEGRADE_TAB_INTS words");

// Reverb (or a plain copy for variants without it): CTA (tile, k) writes outputs [o0, o0 + 2048) of variant k,
//   y[o] = sum_{j < L} h[j] x[o - j]   (x = 0 outside [0, n)).
// Thread t accumulates the 8 consecutive outputs o0 + 8t + r in registers.  Taps go in groups of 4: the 32 products of a group read
// the 12 samples x[o0 + 8t - j - 4 .. + 8); the group after it needs 4 new samples, one 16-byte shared load, and the 4 taps are one
// broadcast 16-byte load.  Chunks of taps whose samples all lie before x[0] are skipped.
__global__ void __launch_bounds__(FIR_THREADS) fir_reverb_kernel(const float* __restrict__ x, int64_t n, const VarTab* __restrict__ tab,
                                                                const float* __restrict__ taps, float* __restrict__ out) {
  __shared__ __align__(16) float xs[FIR_TJ + FIR_TO + 4];
  __shared__ __align__(16) float hs[FIR_TJ];
  const VarTab v = tab[blockIdx.y];
  const int64_t o0 = (int64_t)blockIdx.x * FIR_TO;
  float* y = out + (int64_t)blockIdx.y * n;
  const int t = threadIdx.x;
  if (!(v.stages & LSD_AD_REVERB)) {
    for (int e = t; e < FIR_TO; e += FIR_THREADS)
      if (o0 + e < n) y[o0 + e] = x[o0 + e];
    return;
  }
  const float* h = taps + v.rir_off;
  const int L = v.rir_len;
  const int j_end = (int)(L < o0 + FIR_TO ? L : o0 + FIR_TO);
  float acc[FIR_R];
#pragma unroll
  for (int r = 0; r < FIR_R; ++r) acc[r] = 0.f;
  for (int j0 = 0; j0 < j_end; j0 += FIR_TJ) {
    __syncthreads();
    for (int q = t; q < FIR_TJ; q += FIR_THREADS) hs[q] = j0 + q < L ? h[j0 + q] : 0.f;
    const int64_t xb = o0 - j0 - FIR_TJ - 4;   // xs[p] = x[xb + p]
    for (int p = t; p < FIR_TJ + FIR_TO + 4; p += FIR_THREADS) {
      const int64_t i = xb + p;
      xs[p] = i >= 0 && i < n ? x[i] : 0.f;
    }
    __syncthreads();
    // w[m] = x[o0 + 8t - jj - 4 + m] = xs[8t + TJ - jj + m] for the group of taps jj .. jj+3 of this chunk
    float w[12];
    const float4* x4 = reinterpret_cast<const float4*>(xs + 8 * t + FIR_TJ);
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const float4 a = x4[q];
      w[4 * q] = a.x; w[4 * q + 1] = a.y; w[4 * q + 2] = a.z; w[4 * q + 3] = a.w;
    }
    const int jn = (j_end - j0) < FIR_TJ ? (j_end - j0) : FIR_TJ;
#pragma unroll 2
    for (int jj = 0; jj < jn; jj += 4) {
      const float4 hv = *reinterpret_cast<const float4*>(hs + jj);
      const float hd[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
      for (int d = 0; d < 4; ++d)
#pragma unroll
        for (int r = 0; r < FIR_R; ++r) acc[r] = fmaf(hd[d], w[r - d + 4], acc[r]);
#pragma unroll
      for (int m = 11; m >= 4; --m) w[m] = w[m - 4];
      const float4 a = *reinterpret_cast<const float4*>(xs + 8 * t + FIR_TJ - jj - 4);
      w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
    }
  }
#pragma unroll
  for (int r = 0; r < FIR_R; ++r)
    if (o0 + 8 * t + r < n) y[o0 + 8 * t + r] = acc[r];
}

__device__ __forceinline__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
  __syncthreads();
  return s;
}

// Noise stage, pass 1: per variant with noise, POW_BLOCKS partial sums of x^2 (the signal as it stands) and g^2, fp64.
__global__ void __launch_bounds__(256) noise_power_kernel(const float* __restrict__ y_all, int64_t n, const VarTab* __restrict__ tab,
                                                          double* __restrict__ part) {
  __shared__ double red[8];
  const VarTab v = tab[blockIdx.y];
  if (!(v.stages & LSD_AD_NOISE)) return;
  const float* y = y_all + (int64_t)blockIdx.y * n;
  const uint64_t key = stream_key(v.seed, 0);
  double sx = 0, sg = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double a = y[i], g = gauss(key, (uint64_t)i);
    sx += a * a;
    sg += g * g;
  }
  sx = block_sum(sx, red);
  sg = block_sum(sg, red);
  if (threadIdx.x == 0) {
    part[((int64_t)blockIdx.y * POW_BLOCKS + blockIdx.x) * 2] = sx;
    part[((int64_t)blockIdx.y * POW_BLOCKS + blockIdx.x) * 2 + 1] = sg;
  }
}

// Noise stage, pass 2, and the clip stage: y = x + s g (s from the partial sums, summed in order), then the clamp.
__global__ void __launch_bounds__(256) noise_clip_kernel(float* __restrict__ y_all, int64_t n, const VarTab* __restrict__ tab,
                                                         const double* __restrict__ part) {
  __shared__ double s_sh;
  const VarTab v = tab[blockIdx.y];
  const bool noise = v.stages & LSD_AD_NOISE, clip = v.stages & LSD_AD_CLIP;
  if (!noise && !clip) return;
  if (threadIdx.x == 0) {
    double s = 0;
    if (noise) {
      double px = 0, pg = 0;
      for (int b = 0; b < POW_BLOCKS; ++b) {
        px += part[((int64_t)blockIdx.y * POW_BLOCKS + b) * 2];
        pg += part[((int64_t)blockIdx.y * POW_BLOCKS + b) * 2 + 1];
      }
      px /= (double)n;
      pg /= (double)n;
      s = px == 0.0 ? 0.0 : sqrt(px / (pg * v.snr_lin));   // a silent clip passes unchanged
    }
    s_sh = s;
  }
  __syncthreads();
  const double s = s_sh;
  const uint64_t key = stream_key(v.seed, 0);
  float* y = y_all + (int64_t)blockIdx.y * n;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float a = y[i];
    if (noise && s != 0.0) a = (float)((double)a + s * gauss(key, (uint64_t)i));
    if (clip) a = fminf(fmaxf(__fmul_rn(a, v.gain), -1.f), 1.f);
    y[i] = a;
  }
}

// Band stage, one pass of resample_poly for the variants with factor f:
//   out[o] = sum_m h[m] x_up[(o + pre) down - pad - m],  x_up[t] = x[t / up] when up divides t, else 0,
// h the host's taps (firwin, scaled by up); o < n_out.  Pass 1: x = the variant's row, up 1, down f, out = its row of `mid`.
// Pass 2: x = that row of `mid`, up f, down 1, out = the variant's row, cut to n.
__global__ void __launch_bounds__(256) upfirdn_kernel(const float* __restrict__ x_all, int64_t n_in, float* __restrict__ out_all,
                                                      int64_t n_out, const VarTab* __restrict__ tab, int f, const float* __restrict__ h,
                                                      int M, int up, int down, int pre, int pad) {
  __shared__ float hs[128];
  if (tab[blockIdx.y].f != f) return;
  for (int m = threadIdx.x; m < M; m += blockDim.x) hs[m] = h[m];
  __syncthreads();
  const float* x = x_all + (int64_t)blockIdx.y * n_in;
  float* out = out_all + (int64_t)blockIdx.y * n_out;
  for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < n_out; o += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t0 = (o + pre) * down - pad;
    int m = (int)(((t0 % up) + up) % up);
    float acc = 0.f;
    for (; m < M; m += up) {
      const int64_t q = (t0 - m) / up;
      if (q >= 0 && q < n_in) acc = fmaf(hs[m], x[q], acc);
    }
    out[o] = acc;
  }
}

// audioop's st_14linear2ulaw / st_ulaw2linear16 (Sun G.711 reference code)
__device__ __forceinline__ int ulaw_round_trip(int s16) {
  int v = s16 >> 2;
  int mask = 0xFF;
  if (v < 0) { v = -v; mask = 0x7F; }
  if (v > 8159) v = 8159;
  v += 0x84 >> 2;
  int seg = 0;
  while (seg < 8 && v > (0x40 << seg) - 1) ++seg;   // seg_uend[seg] = 0x3F, 0x7F, 0xFF, ... 0x1FFF
  int u = seg >= 8 ? 0x7F : ((seg << 4) | ((v >> (seg + 1)) & 0xF));
  u = (~(u ^ mask)) & 0xFF;
  int tt = (((u & 0x0F) << 3) + 0x84) << ((u & 0x70) >> 4);
  return (u & 0x80) ? 0x84 - tt : tt - 0x84;
}

__global__ void __launch_bounds__(256) mulaw_kernel(float* __restrict__ y_all, int64_t n, const VarTab* __restrict__ tab) {
  if (!(tab[blockIdx.y].stages & LSD_AD_MULAW)) return;
  float* y = y_all + (int64_t)blockIdx.y * n;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float r = rintf(__fmul_rn(y[i], 32768.f));
    const int s = (int)fminf(fmaxf(r, -32768.f), 32767.f);
    y[i] = __fdiv_rn((float)ulaw_round_trip(s), 32768.f);
  }
}

// firwin(20 f + 1, 1 / f, window=('kaiser', 5.0)) in double: sinc lowpass times the Kaiser window, scaled to unit DC gain
double bessel_i0(double x) {
  double s = 1, term = 1;
  for (int k = 1; k < 200; ++k) {
    term *= (x / (2.0 * k)) * (x / (2.0 * k));
    s += term;
    if (term < 1e-17 * s) break;
  }
  return s;
}
void kaiser_lowpass(int f, std::vector<double>& h) {
  const int M = 20 * f + 1;
  const double alpha = (M - 1) / 2.0, cutoff = 1.0 / f, pi = 3.141592653589793;
  h.assign(M, 0.0);
  double sum = 0;
  for (int i = 0; i < M; ++i) {
    const double m = i - alpha, a = cutoff * m;
    const double sinc = a == 0.0 ? 1.0 : sin(pi * a) / (pi * a);
    const double r = (i - alpha) / alpha;
    h[i] = cutoff * sinc * bessel_i0(5.0 * sqrt(1.0 - r * r)) / bessel_i0(5.0);
    sum += h[i];
  }
  for (double& v : h) v /= sum;
}

int grid_for(int64_t n, int per_block) {
  const int64_t b = (n + per_block - 1) / per_block;
  return (int)(b < 2048 ? b : 2048);
}

}  // namespace

int degrade_rir_length(float rt60) { return (int)nearbyint((double)rt60 * SR); }

// Host half: the device table (K VarTab, the band taps of f = 2 and 4 for both passes, the impulse responses) as int32 words.
void degrade_tables(const lsd_audio_degradation* v, int K, std::vector<int32_t>& out) {
  std::vector<float> band;
  for (int f : {2, 4}) {
    std::vector<double> h;
    kaiser_lowpass(f, h);
    for (int pass = 0; pass < 2; ++pass)
      for (double t : h) band.push_back((float)(pass ? t * f : t));
  }
  int rir_total = 0;
  for (int k = 0; k < K; ++k)
    if (v[k].stages & LSD_AD_REVERB) rir_total += degrade_rir_length(v[k].rt60);
  const size_t tab_words = (size_t)K * DEGRADE_TAB_INTS;
  out.assign(tab_words + band.size() + rir_total, 0);
  memcpy(out.data() + tab_words, band.data(), band.size() * sizeof(float));
  float* rir = reinterpret_cast<float*>(out.data() + tab_words + band.size());
  int off = (int)band.size();   // floats past the table
  for (int k = 0; k < K; ++k) {
    VarTab t{};
    t.stages = v[k].stages;
    t.seed = v[k].seed;
    if (v[k].stages & LSD_AD_REVERB) {
      const int L = degrade_rir_length(v[k].rt60);
      const uint64_t key = stream_key(v[k].seed, 1);
      std::vector<double> tail(L);
      double e = 0;
      for (int j = 1; j < L; ++j) {
        tail[j] = gauss(key, (uint64_t)j) * pow(10.0, -3.0 * (double)j / L);
        e += tail[j] * tail[j];
      }
      const double sc = 1.0 / sqrt(e);
      rir[off - (int)band.size()] = 1.f;
      for (int j = 1; j < L; ++j) rir[off - (int)band.size() + j] = (float)(tail[j] * sc);
      t.rir_len = L;
      t.rir_off = off;
      off += L;
    }
    if (v[k].stages & LSD_AD_NOISE) t.snr_lin = pow(10.0, (double)v[k].snr_db / 10.0);
    if (v[k].stages & LSD_AD_CLIP) t.gain = (float)pow(10.0, (double)v[k].gain_db / 20.0);
    if (v[k].stages & LSD_AD_BAND) t.f = SR / v[k].band_rate;
    memcpy(out.data() + (size_t)k * DEGRADE_TAB_INTS, &t, sizeof(t));
  }
}

size_t degrade_partials_bytes(int K) { return (size_t)K * POW_BLOCKS * 2 * sizeof(double); }

// Device half.  tab: degrade_tables as copied to the device; part: degrade_partials_bytes; mid: K * ceil(n / 2) floats.
void launch_degrade_audio(const float* pcm, int64_t n, const lsd_audio_degradation* v, int K, const int32_t* tab, double* part,
                          float* mid, float* out, cudaStream_t s) {
  const VarTab* vt = reinterpret_cast<const VarTab*>(tab);
  const float* band = reinterpret_cast<const float*>(tab + (size_t)K * DEGRADE_TAB_INTS);
  int any = 0;
  for (int k = 0; k < K; ++k) any |= v[k].stages;
  fir_reverb_kernel<<<dim3((unsigned)((n + FIR_TO - 1) / FIR_TO), K), FIR_THREADS, 0, s>>>(pcm, n, vt, band, out);
  int launches = 1;
  if (any & LSD_AD_NOISE) {
    noise_power_kernel<<<dim3(POW_BLOCKS, K), 256, 0, s>>>(out, n, vt, part);
    ++launches;
  }
  if (any & (LSD_AD_NOISE | LSD_AD_CLIP)) {
    noise_clip_kernel<<<dim3(grid_for(n, 1024), K), 256, 0, s>>>(out, n, vt, part);
    ++launches;
  }
  int h_off = 0;
  for (int f : {2, 4}) {
    const int M = 20 * f + 1;
    bool used = false;
    for (int k = 0; k < K; ++k) used |= (v[k].stages & LSD_AD_BAND) && SR / v[k].band_rate == f;
    if (used) {
      const int64_t n_mid = (n + f - 1) / f;
      const int half = 10 * f;
      // resample_poly's zero padding in front of the taps and the samples it drops: (up 1, down f), then (up f, down 1)
      const int pad1 = f - half % f, pre1 = (half + pad1) / f, pad2 = 1, pre2 = half + 1;
      upfirdn_kernel<<<dim3(grid_for(n_mid, 256), K), 256, 0, s>>>(out, n, mid, n_mid, vt, f, band + h_off, M, 1, f, pre1, pad1);
      upfirdn_kernel<<<dim3(grid_for(n, 256), K), 256, 0, s>>>(mid, n_mid, out, n, vt, f, band + h_off + M, M, f, 1, pre2, pad2);
      launches += 2;
    }
    h_off += 2 * M;
  }
  if (any & LSD_AD_MULAW) {
    mulaw_kernel<<<dim3(grid_for(n, 1024), K), 256, 0, s>>>(out, n, vt);
    ++launches;
  }
  count_launch(launches);
}

}  // namespace lsd
