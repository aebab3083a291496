// Small fp32 kernels of the token path on the bf16 (tensor-core) route.  They keep LayerNorm / softmax / gating / the
// head in fp32 (SURVEY.md §7.3 bf16 budget) and hand their results to the tcgen05 GEMMs as padded planar bf16.
// Reference semantics: fusion_module.py:54-87, temporal.py:64-111, artifact_detector.py:142-181, classifier.py:14-34.
#include "token_kernels.cuh"

#include <math.h>

namespace lsd {

__device__ __forceinline__ int64_t pmap(const PlanarOut& o, int64_t row) {
  return o.grp > 0 ? (row / o.grp) * o.grp_stride + (row % o.grp) + o.off : row + o.off;
}
__device__ __forceinline__ void pstore(const PlanarOut& o, int64_t pos, int c, float v) {
  const int64_t idx = (int64_t)(c >> 3) * o.plane_stride + pos * 8 + (c & 7);
  const __nv_bfloat16 hi = __float2bfloat16_rn(v);
  o.y[idx] = hi;
  if (o.ylo) o.ylo[idx] = __float2bfloat16_rn(v - __bfloat162float(hi));
}
__device__ __forceinline__ float tk_warp_sum(float v) {
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}
__device__ __forceinline__ float tk_warp_max(float v) {
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, s));
  return v;
}
__device__ __forceinline__ float tk_gelu(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// ---- LayerNorm (eps 1e-5), fp32 in -> planar bf16 out; one warp per row
__global__ void layernorm_p_kernel(const float* x, int64_t x_ld, const float* g, const float* b, int rows, int D, PlanarOut o) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + (int64_t)row * x_ld;
  float s = 0.f;
  for (int d = lane; d < D; d += 32) s += xr[d];
  const float mu = tk_warp_sum(s) / (float)D;
  float v = 0.f;
  for (int d = lane; d < D; d += 32) { const float t = xr[d] - mu; v += t * t; }
  const float rstd = 1.0f / sqrtf(tk_warp_sum(v) / (float)D + 1e-5f);
  const int64_t pos = pmap(o, row);
  for (int d = lane; d < D; d += 32) pstore(o, pos, d, (xr[d] - mu) * rstd * g[d] + b[d]);
}
void launch_layernorm_p(const float* x, int64_t x_ld, const float* g, const float* b, int rows, int D, PlanarOut o, cudaStream_t s) {
  if (rows == 0) return;
  layernorm_p_kernel<<<(rows + 7) / 8, 256, 0, s>>>(x, x_ld, g, b, rows, D, o);
  count_launch();
}

// ---- attention core (head dim 32), fp32 q/k/v rows -> planar bf16 (and/or fp32) output
__global__ void mha_core_p_kernel(const float* q, int q_ld, const float* k, int k_ld, const float* v, int v_ld, int Tq, int Tk, int heads,
                                  PlanarOut o) {
  extern __shared__ float sm[];
  float* Ks = sm;
  float* Vs = sm + (size_t)Tk * 33;
  const int n = blockIdx.x / heads, h = blockIdx.x % heads;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int j = warp; j < Tk; j += nwarps) {
    Ks[j * 33 + lane] = k[((int64_t)n * Tk + j) * k_ld + h * 32 + lane];
    Vs[j * 33 + lane] = v[((int64_t)n * Tk + j) * v_ld + h * 32 + lane];
  }
  __syncthreads();
  const float scale = 0.17677669529663688f;  // 1/sqrt(32)
  for (int i = warp; i < Tq; i += nwarps) {
    const float qd = q[((int64_t)n * Tq + i) * q_ld + h * 32 + lane] * scale;
    float acc = 0.f, mx = -INFINITY, den = 0.f;
    for (int j0 = 0; j0 < Tk; j0 += 32) {
      const int j = j0 + lane;
      float dot = 0.f;
#pragma unroll
      for (int d = 0; d < 32; ++d) {
        const float qv = __shfl_sync(0xffffffffu, qd, d);
        if (j < Tk) dot = fmaf(qv, Ks[j * 33 + d], dot);
      }
      mx = fmaxf(mx, tk_warp_max(j < Tk ? dot : -INFINITY));
    }
    for (int j0 = 0; j0 < Tk; j0 += 32) {
      const int j = j0 + lane;
      float dot = 0.f;
#pragma unroll
      for (int d = 0; d < 32; ++d) {
        const float qv = __shfl_sync(0xffffffffu, qd, d);
        if (j < Tk) dot = fmaf(qv, Ks[j * 33 + d], dot);
      }
      const float pj = (j < Tk) ? expf(dot - mx) : 0.f;
      den += tk_warp_sum(pj);
      const int cnt = min(32, Tk - j0);
      for (int jj = 0; jj < cnt; ++jj) acc = fmaf(__shfl_sync(0xffffffffu, pj, jj), Vs[(j0 + jj) * 33 + lane], acc);
    }
    pstore(o, pmap(o, (int64_t)n * Tq + i), h * 32 + lane, acc / den);
  }
}
// Register-resident variant for Tk <= 64 (every shape of this model: 16/17/32/33 keys): K and V of one (window, head) are
// staged in shared memory with coalesced loads; lane j keeps key rows j and j+32 in registers, a query row is broadcast from
// shared memory (LDS.128), so Q.K^T costs one FMA per (key, dim) with no shuffles; softmax statistics by warp reduction;
// P.V broadcasts p_j by shuffle against V rows in shared memory (lane = output dim).
__global__ void __launch_bounds__(128) mha_core_p64_kernel(const float* __restrict__ q, int q_ld, const float* __restrict__ k, int k_ld,
                                                           const float* __restrict__ v, int v_ld, int Tq, int Tk, int heads, PlanarOut o) {
  extern __shared__ __align__(16) float sm[];
  float* Qs = sm;                                // [Tq][32], pre-scaled (first: rows stay 16-byte aligned for LDS.128)
  float* Ks = Qs + (size_t)Tq * 32;              // [Tk][33]
  float* Vs = Ks + (size_t)Tk * 33;              // [Tk][33]
  const int n = blockIdx.x / heads, h = blockIdx.x % heads;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const float scale = 0.17677669529663688f;  // 1/sqrt(32)
  for (int j = warp; j < Tk; j += nwarps) {
    Ks[j * 33 + lane] = k[((int64_t)n * Tk + j) * k_ld + h * 32 + lane];
    Vs[j * 33 + lane] = v[((int64_t)n * Tk + j) * v_ld + h * 32 + lane];
  }
  for (int i = warp; i < Tq; i += nwarps) Qs[i * 32 + lane] = q[((int64_t)n * Tq + i) * q_ld + h * 32 + lane] * scale;
  __syncthreads();
  const bool two = Tk > 32;
  const bool v0 = lane < Tk, v1 = lane + 32 < Tk;
  float k0[32], k1[32];
#pragma unroll
  for (int d = 0; d < 32; ++d) {
    k0[d] = v0 ? Ks[lane * 33 + d] : 0.f;
    k1[d] = v1 ? Ks[(lane + 32) * 33 + d] : 0.f;
  }
  for (int i = warp; i < Tq; i += nwarps) {
    float d0 = 0.f, d1 = 0.f;
    const float4* qr = reinterpret_cast<const float4*>(Qs + i * 32);
#pragma unroll
    for (int d4 = 0; d4 < 8; ++d4) {
      const float4 qv = qr[d4];
      d0 = fmaf(qv.x, k0[4 * d4], d0); d0 = fmaf(qv.y, k0[4 * d4 + 1], d0); d0 = fmaf(qv.z, k0[4 * d4 + 2], d0); d0 = fmaf(qv.w, k0[4 * d4 + 3], d0);
      if (two) { d1 = fmaf(qv.x, k1[4 * d4], d1); d1 = fmaf(qv.y, k1[4 * d4 + 1], d1); d1 = fmaf(qv.z, k1[4 * d4 + 2], d1); d1 = fmaf(qv.w, k1[4 * d4 + 3], d1); }
    }
    const float mx = tk_warp_max(fmaxf(v0 ? d0 : -INFINITY, v1 ? d1 : -INFINITY));
    const float p0 = v0 ? expf(d0 - mx) : 0.f, p1 = v1 ? expf(d1 - mx) : 0.f;
    // fixed summation order (the same as the generic kernel: tile 0 then tile 1)
    const float den = tk_warp_sum(p0) + (two ? tk_warp_sum(p1) : 0.f);
    float acc = 0.f;
    const int c0 = min(32, Tk);
    for (int j = 0; j < c0; ++j) acc = fmaf(__shfl_sync(0xffffffffu, p0, j), Vs[j * 33 + lane], acc);
    for (int j = 32; j < Tk; ++j) acc = fmaf(__shfl_sync(0xffffffffu, p1, j - 32), Vs[j * 33 + lane], acc);
    pstore(o, pmap(o, (int64_t)n * Tq + i), h * 32 + lane, acc / den);
  }
}
void launch_mha_core_p(const float* q, int q_ld, const float* k, int k_ld, const float* v, int v_ld, int N, int Tq, int Tk, int heads,
                       PlanarOut o, cudaStream_t s) {
  if (N == 0) return;
  if (Tk <= 64)
    mha_core_p64_kernel<<<N * heads, 128, ((size_t)Tk * 33 * 2 + (size_t)Tq * 32) * sizeof(float), s>>>(q, q_ld, k, k_ld, v, v_ld, Tq, Tk, heads, o);
  else
    mha_core_p_kernel<<<N * heads, 128, (size_t)Tk * 33 * 2 * sizeof(float), s>>>(q, q_ld, k, k_ld, v, v_ld, Tq, Tk, heads, o);
  count_launch();
}

// ---- gate: g = sigmoid(h . w2 + b2); out = g*v + (1-g)*a  -> planar bf16
__global__ void gate_blend_p_kernel(const float* h, const float* w2, const float* b2, const float* v, int v_ld, const float* a, int a_ld,
                                    int rows, int D, PlanarOut o) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float s = 0.f;
  for (int d = lane; d < D; d += 32) s = fmaf(h[(int64_t)row * D + d], w2[d], s);
  s = tk_warp_sum(s) + b2[0];
  const float g = 1.0f / (1.0f + expf(-s));
  const int64_t pos = pmap(o, row);
  for (int d = lane; d < D; d += 32) pstore(o, pos, d, g * v[(int64_t)row * v_ld + d] + (1.0f - g) * a[(int64_t)row * a_ld + d]);
}
void launch_gate_blend_p(const float* h, const float* w2, const float* b2, const float* v, int v_ld, const float* a, int a_ld, int rows,
                         int D, PlanarOut o, cudaStream_t s) {
  if (rows == 0) return;
  gate_blend_p_kernel<<<(rows + 7) / 8, 256, 0, s>>>(h, w2, b2, v, v_ld, a, a_ld, rows, D, o);
  count_launch();
}

// ---- F.interpolate(linear, align_corners=False) over tokens: fp32 rows (residual) + planar bf16 (GEMM input)
__global__ void lerp_tokens_p_kernel(const float* x, float* y, int Tin, int Tout, int D, int64_t total, PlanarOut o) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int d = (int)(i % D);
  const int64_t r = i / D;
  const int t = (int)(r % Tout);
  const int64_t n = r / Tout;
  float val;
  if (Tin == Tout) {
    val = x[i];
  } else {
    const float scale = (float)Tin / (float)Tout;
    float src = ((float)t + 0.5f) * scale - 0.5f;
    src = src < 0.f ? 0.f : src;
    int i0 = (int)floorf(src);
    i0 = i0 > Tin - 1 ? Tin - 1 : i0;
    const int i1 = i0 + 1 > Tin - 1 ? Tin - 1 : i0 + 1;
    const float w1 = src - (float)i0;
    const float* b = x + n * (int64_t)Tin * D + d;
    val = b[(int64_t)i0 * D] * (1.0f - w1) + b[(int64_t)i1 * D] * w1;
  }
  if (y) y[i] = val;
  pstore(o, pmap(o, r), d, val);
}
void launch_lerp_tokens_p(const float* x, float* y, int N, int Tin, int Tout, int D, PlanarOut o, cudaStream_t s) {
  const int64_t total = (int64_t)N * Tout * D;
  if (total == 0) return;
  lerp_tokens_p_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(x, y, Tin, Tout, D, total, o);
  count_launch();
}

// ---- log-mel window (N,1,F,Ta) of any float dtype -> bf16 "pixel rows" for the Toeplitz audio stem.
// Each sample occupies one 4-channel pixel: ch0 = hi = bf16(x), ch1 = lo = bf16(x - hi), ch2 = hi, ch3 = 0; the stem weights
// are (W_hi, W_hi, W_lo, 0), i.e. x*W ~ hi*W_hi + lo*W_hi + hi*W_lo (split-bf16: ~16 mantissa bits of both operands).
__global__ void audio_rows_kernel(const void* audio, int dtype, __nv_bfloat16* y, int64_t set_stride, UcGeom g, int F, int Ta, int64_t total) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int WP = (Ta + 1) / 2;
  const int wp = (int)(i % WP);
  int64_t r = i / WP;
  const int f = (int)(r % F);
  const int n = (int)(r / F);
  __nv_bfloat16 px[8];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int a = 2 * wp + q;
    float x = 0.f;
    if (a < Ta) {
      const int64_t idx = ((int64_t)n * F + f) * Ta + a;
      x = dtype == 0 ? reinterpret_cast<const float*>(audio)[idx]
                     : (dtype == 1 ? __half2float(reinterpret_cast<const __half*>(audio)[idx])
                                   : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(audio)[idx]));
    }
    const __nv_bfloat16 hi = __float2bfloat16_rn(x);
    px[q * 4 + 0] = hi;
    px[q * 4 + 1] = __float2bfloat16_rn(x - __bfloat162float(hi));
    px[q * 4 + 2] = hi;
    px[q * 4 + 3] = __float2bfloat16_rn(0.f);
  }
  const int64_t flat = (((int64_t)n * g.TS + g.ot) * g.HP + (f >> 1) + g.oh) * g.RW + g.ow;
  const int64_t dst = (int64_t)(f & 1) * set_stride + flat * 8 + (int64_t)(2 * wp + 4) * 4;
  *reinterpret_cast<uint4*>(y + dst) = *reinterpret_cast<const uint4*>(px);
}
void launch_audio_rows(const void* audio, int dtype, __nv_bfloat16* y, int64_t set_stride, UcGeom g, int F, int Ta, cudaStream_t s) {
  const int64_t total = (int64_t)g.N * F * ((Ta + 1) / 2);
  if (total == 0) return;
  audio_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(audio, dtype, y, set_stride, g, F, Ta, total);
  count_launch();
}

// ---- fused head: artifact fusion MLP (448->256 ReLU ->128 ReLU), cat[cls|artifact], Linear 384->128, GELU, LayerNorm(128),
// Linear 128->1.  One block (256 threads) per window, everything in fp32, weights [Cin][Cout] from the fp32 arena.
// 512 threads: every layer splits its K range over 2 (448 -> 256) or 4 (256 -> 128, 384 -> 128) thread groups and keeps 16
// independent weight loads in flight per thread — the kernel is L2-latency-bound (0.9 MB of fp32 weights per window, one
// window per SM); partial sums are combined in a fixed order.
// cls: row n of the CLS outputs at cls + n * cls_ld (read in place from the token buffer); comb[:, 256:448]: artifact features,
// row n / K (K audio variants of one video share its artifact features; K = 1: one row per window).
__global__ void __launch_bounds__(512) head_kernel(const float* __restrict__ cls, int64_t cls_ld, const float* __restrict__ comb, HeadW w,
                                                   float* __restrict__ logits, int K) {
  __shared__ float x[448], h1[256], f[384], part[512], red[4];
  const int n = blockIdx.x, tid = threadIdx.x;
  const int64_t crow = n / K;
  for (int i = tid; i < 448; i += 512) x[i] = i < 256 ? cls[(int64_t)n * cls_ld + i] : comb[crow * 448 + i];
  __syncthreads();
  {
    const int o = tid & 255, half = tid >> 8;                 // K split: [0,224) and [224,448)
    const float* wp = w.w0 + (size_t)half * 224 * 256 + o;
    const float* xp = x + half * 224;
    float acc = 0.f;
#pragma unroll 16
    for (int k = 0; k < 224; ++k) acc = fmaf(xp[k], wp[(size_t)k * 256], acc);
    part[tid] = acc;
  }
  __syncthreads();
  if (tid < 256) { h1[tid] = fmaxf(w.b0[tid] + part[tid] + part[tid + 256], 0.f); f[tid] = x[tid]; }   // f[0:256] = cls
  __syncthreads();
  {
    const int o = tid & 127, q = tid >> 7;                    // K split: 4 x 64
    const float* wp = w.w2 + (size_t)q * 64 * 128 + o;
    const float* xp = h1 + q * 64;
    float acc = 0.f;
#pragma unroll 16
    for (int k = 0; k < 64; ++k) acc = fmaf(xp[k], wp[(size_t)k * 128], acc);
    part[tid] = acc;
  }
  __syncthreads();
  if (tid < 128) f[256 + tid] = fmaxf(w.b2[tid] + ((part[tid] + part[tid + 128]) + (part[tid + 256] + part[tid + 384])), 0.f);
  __syncthreads();
  {
    const int o = tid & 127, q = tid >> 7;                    // K split: 4 x 96
    const float* wp = w.wc + (size_t)q * 96 * 128 + o;
    const float* xp = f + q * 96;
    float acc = 0.f;
#pragma unroll 16
    for (int k = 0; k < 96; ++k) acc = fmaf(xp[k], wp[(size_t)k * 128], acc);
    part[tid] = acc;
  }
  __syncthreads();
  float hv = 0.f;
  if (tid < 128) hv = tk_gelu(w.bc[tid] + ((part[tid] + part[tid + 128]) + (part[tid + 256] + part[tid + 384])));
  // LayerNorm(128) + dot, fixed-order reductions over the first four warps
  float s = (tid < 128) ? hv : 0.f;
  s = tk_warp_sum(s);
  if (tid < 128 && (tid & 31) == 0) red[tid >> 5] = s;
  __syncthreads();
  const float mu = (red[0] + red[1] + red[2] + red[3]) / 128.0f;
  __syncthreads();
  float d = (tid < 128) ? (hv - mu) * (hv - mu) : 0.f;
  d = tk_warp_sum(d);
  if (tid < 128 && (tid & 31) == 0) red[tid >> 5] = d;
  __syncthreads();
  const float rstd = 1.0f / sqrtf((red[0] + red[1] + red[2] + red[3]) / 128.0f + 1e-5f);
  __syncthreads();
  float o = (tid < 128) ? ((hv - mu) * rstd * w.lng[tid] + w.lnb[tid]) * w.wo[tid] : 0.f;
  o = tk_warp_sum(o);
  if (tid < 128 && (tid & 31) == 0) red[tid >> 5] = o;
  __syncthreads();
  if (tid == 0) logits[n] = red[0] + red[1] + red[2] + red[3] + w.bo[0];
}
void launch_head(const float* cls, int64_t cls_ld, const float* comb, const HeadW& w, float* logits, int B, cudaStream_t s, int K) {
  if (B == 0) return;
  head_kernel<<<B, 512, 0, s>>>(cls, cls_ld, comb, w, logits, K);
  count_launch();
}

}  // namespace lsd
