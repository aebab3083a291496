// Branch attribution (lsd_branch_attribution): exact Shapley values of the classifier head's four inputs, sync = cls[0:256],
// raw = [256:320], delta = [320:384], hf = [384:448] of the head's 448-wide input row, against a background set of M rows.
// Player p is bit p of a coalition mask S; the hybrid row x^{S,j} takes slice p from the window row when bit p is set and from
// background row j otherwise, and v(S) = (1/M) sum_j f(x^{S,j}) with f the head in logit space.
//
// The head's first layer is linear, so W0^T x = sum_p W0_p^T x_p: branch_project_kernel computes, once per window row and once per
// background row, P_p = W0_p^T x_p (4 x 256) and C = Wc[0:256]^T cls (128; the head's fc0 reads cls directly).  A hybrid row
// then only costs the tail: h1 = relu(b0 + P_sync + P_raw + P_delta + P_hf), a = relu(b2 + W2^T h1), z = bc + C + Wc[256:384]^T a,
// GELU, LayerNorm(128), dot with head.out (coalition_tail_kernel), ~49k MAC against ~197k for the whole head.
//
// Everything is fp32 FFMA (no tensor cores): Shapley values are differences of neighbouring coalition values, and TF32 / bf16
// operands would put ~1e-3 relative error on each of them.  Bits: every row is computed by the same instruction sequence whatever
// its position in a tile, its window's index or the number of windows; the sum over a background chunk is taken in j order and the
// chunks are summed in chunk order, and the chunking depends on M only.  So the results do not depend on n or on how windows are
// split over calls, and identical hybrid rows give identical logits (a background equal to the window gives phi == 0 exactly).
#include "lsd_kernels.h"
#include "token_kernels.cuh"

#include <algorithm>

namespace lsd {
namespace {

constexpr int PROJ_ROWS = 8;                       // rows per block of branch_project_kernel
constexpr int TAIL_THREADS = 256;
constexpr int TAIL_ROWS = 32;                      // hybrid rows per tile: 15 masks x ATTR_CHUNK backgrounds, S = 15, one pad row
constexpr int TAIL_SMEM_FLOATS = 256 * 128 + 128 * 128 + TAIL_ROWS * 256 + TAIL_ROWS;

// GELU (erf), rounded op by op so that no row can be contracted differently from another
__device__ __forceinline__ float attr_gelu(float x) {
  return __fmul_rn(__fmul_rn(0.5f, x), __fadd_rn(1.0f, erff(__fmul_rn(x, 0.70710678118654752f))));
}

// Sum over the 16 lanes of a half warp (lanes 0..15 or 16..31), the same tree for every half.
__device__ __forceinline__ float half_warp_sum(float v) {
#pragma unroll
  for (int s = 8; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}

// Row r < n: window row r of feats, else background row r - n.  One block of 256 threads per PROJ_ROWS rows; thread o owns output
// column o of every slice and keeps one accumulator per row, k ascending within the slice.
__global__ void __launch_bounds__(256) branch_project_kernel(const float* __restrict__ feats, int n, const float* __restrict__ bg, int M,
                                                             HeadW w, float* __restrict__ proj) {
  __shared__ float x[PROJ_ROWS][LSD_BRANCH_FEATURES];
  const int r0 = blockIdx.x * PROJ_ROWS, R = n + M, tid = threadIdx.x;
  for (int e = tid; e < PROJ_ROWS * LSD_BRANCH_FEATURES; e += 256) {
    const int q = e / LSD_BRANCH_FEATURES, c = e - q * LSD_BRANCH_FEATURES, r = r0 + q;
    float v = 0.f;
    if (r < n) v = feats[(int64_t)r * LSD_BRANCH_FEATURES + c];
    else if (r < R) v = bg[(int64_t)(r - n) * LSD_BRANCH_FEATURES + c];
    x[q][c] = v;
  }
  __syncthreads();
  const int o = tid;
  const int k_lo[4] = {0, 256, 320, 384}, k_hi[4] = {256, 320, 384, 448};
#pragma unroll 1
  for (int p = 0; p < LSD_BRANCHES; ++p) {
    float acc[PROJ_ROWS];
#pragma unroll
    for (int q = 0; q < PROJ_ROWS; ++q) acc[q] = 0.f;
#pragma unroll 4
    for (int k = k_lo[p]; k < k_hi[p]; ++k) {
      const float wk = w.w0[(size_t)k * 256 + o];
#pragma unroll
      for (int q = 0; q < PROJ_ROWS; ++q) acc[q] = fmaf(x[q][k], wk, acc[q]);
    }
#pragma unroll
    for (int q = 0; q < PROJ_ROWS; ++q)
      if (r0 + q < R) proj[(int64_t)(r0 + q) * ATTR_PROJ + p * 256 + o] = acc[q];
  }
  if (o < 128) {
    float acc[PROJ_ROWS];
#pragma unroll
    for (int q = 0; q < PROJ_ROWS; ++q) acc[q] = 0.f;
#pragma unroll 4
    for (int k = 0; k < 256; ++k) {
      const float wk = w.wc[(size_t)k * 128 + o];
#pragma unroll
      for (int q = 0; q < PROJ_ROWS; ++q) acc[q] = fmaf(x[q][k], wk, acc[q]);
    }
#pragma unroll
    for (int q = 0; q < PROJ_ROWS; ++q)
      if (r0 + q < R) proj[(int64_t)(r0 + q) * ATTR_PROJ + 4 * 256 + o] = acc[q];
  }
}

// Persistent blocks over tiles (window i, background chunk c): tile row r < 30 is (mask r / 2, background j = c*ATTR_CHUNK + r % 2),
// row 30 is S = 15 (the window itself), row 31 pads.  W2 and Wc[256:384] stay in shared memory for the block's lifetime (192 KB);
// the tile's h1 rows (32 KB) are built from the projections and then overwritten by its a rows.  Thread (ty, tx) = (tid / 16,
// tid % 16) owns rows 2ty, 2ty+1 and columns 4tx..4tx+3, 64+4tx..64+4tx+3 of both GEMMs: one accumulator chain per output, k
// ascending.  The LayerNorm and output reductions of a row run over the 16 threads of its half warp.
// partial[(i*15 + S)*n_chunks + c] = the sum of chunk c's logits of mask S in j order; v15[i] = f(x_i).
__global__ void __launch_bounds__(TAIL_THREADS, 1) coalition_tail_kernel(const float* __restrict__ proj, int n, int M, HeadW w,
                                                                         float* __restrict__ partial, float* __restrict__ v15) {
  extern __shared__ float4 smem4[];
  float* sm = reinterpret_cast<float*>(smem4);
  float* W2s = sm;                                  // [256][128]
  float* Wcs = W2s + 256 * 128;                     // [128][128] = Wc rows 256..383
  float* Hs = Wcs + 128 * 128;                      // [32][256] h1, then [32][128] a (row stride 256)
  float* Ls = Hs + TAIL_ROWS * 256;                 // [32] logits of the tile
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  for (int e = tid; e < 256 * 128 / 4; e += TAIL_THREADS) reinterpret_cast<float4*>(W2s)[e] = reinterpret_cast<const float4*>(w.w2)[e];
  for (int e = tid; e < 128 * 128 / 4; e += TAIL_THREADS)
    reinterpret_cast<float4*>(Wcs)[e] = reinterpret_cast<const float4*>(w.wc + 256 * 128)[e];
  const int n_chunks = (M + ATTR_CHUNK - 1) / ATTR_CHUNK;
  const int64_t n_tiles = (int64_t)n * n_chunks;
  const float* pwin_base = proj;
  const float* pbg_base = proj + (int64_t)n * ATTR_PROJ;
  float b2v[8], bcv[8], gv[8], bv[8], wov[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int col = (q < 4 ? 4 * tx + q : 64 + 4 * tx + q - 4);
    b2v[q] = w.b2[col]; bcv[q] = w.bc[col]; gv[q] = w.lng[col]; bv[q] = w.lnb[col]; wov[q] = w.wo[col];
  }
  const float bo = w.bo[0];
  const float b0v = w.b0[tid];
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int i = (int)(tile / n_chunks), c = (int)(tile - (int64_t)i * n_chunks);
    const float* pwin = pwin_base + (int64_t)i * ATTR_PROJ;
    __syncthreads();                                // the previous tile is done with Hs and Ls (and the weights are staged)
    // ---- h1 rows: thread tid owns column tid of every row
#pragma unroll 4
    for (int r = 0; r < TAIL_ROWS; ++r) {
      int mask = 15, j = 0;
      if (r < 30) { mask = r >> 1; j = min(c * ATTR_CHUNK + (r & 1), M - 1); }
      const float* pb = pbg_base + (int64_t)j * ATTR_PROJ;
      float s = b0v;
#pragma unroll
      for (int p = 0; p < LSD_BRANCHES; ++p) s = __fadd_rn(s, ((mask >> p) & 1 ? pwin : pb)[p * 256 + tid]);
      Hs[r * 256 + tid] = fmaxf(s, 0.f);
    }
    __syncthreads();
    // ---- a = relu(b2 + W2^T h1)
    float acc[2][8];
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[u][q] = 0.f;
    {
      const float* h0 = Hs + (2 * ty) * 256;
      const float* h1 = h0 + 256;
#pragma unroll 2
      for (int k = 0; k < 256; k += 4) {
        const float4 a0 = *reinterpret_cast<const float4*>(h0 + k), a1 = *reinterpret_cast<const float4*>(h1 + k);
        const float av0[4] = {a0.x, a0.y, a0.z, a0.w}, av1[4] = {a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const float4 wl = *reinterpret_cast<const float4*>(W2s + (k + kk) * 128 + 4 * tx);
          const float4 wh = *reinterpret_cast<const float4*>(W2s + (k + kk) * 128 + 64 + 4 * tx);
          const float wv[8] = {wl.x, wl.y, wl.z, wl.w, wh.x, wh.y, wh.z, wh.w};
#pragma unroll
          for (int q = 0; q < 8; ++q) { acc[0][q] = fmaf(av0[kk], wv[q], acc[0][q]); acc[1][q] = fmaf(av1[kk], wv[q], acc[1][q]); }
        }
      }
    }
    __syncthreads();                                // every thread is done reading h1
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      float* ar = Hs + (2 * ty + u) * 256;
      *reinterpret_cast<float4*>(ar + 4 * tx) = make_float4(fmaxf(__fadd_rn(b2v[0], acc[u][0]), 0.f), fmaxf(__fadd_rn(b2v[1], acc[u][1]), 0.f),
                                                            fmaxf(__fadd_rn(b2v[2], acc[u][2]), 0.f), fmaxf(__fadd_rn(b2v[3], acc[u][3]), 0.f));
      *reinterpret_cast<float4*>(ar + 64 + 4 * tx) = make_float4(fmaxf(__fadd_rn(b2v[4], acc[u][4]), 0.f), fmaxf(__fadd_rn(b2v[5], acc[u][5]), 0.f),
                                                                 fmaxf(__fadd_rn(b2v[6], acc[u][6]), 0.f), fmaxf(__fadd_rn(b2v[7], acc[u][7]), 0.f));
    }
    __syncthreads();
    // ---- z = bc + C + Wc[256:384]^T a
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[u][q] = 0.f;
    {
      const float* h0 = Hs + (2 * ty) * 256;
      const float* h1 = h0 + 256;
#pragma unroll 2
      for (int k = 0; k < 128; k += 4) {
        const float4 a0 = *reinterpret_cast<const float4*>(h0 + k), a1 = *reinterpret_cast<const float4*>(h1 + k);
        const float av0[4] = {a0.x, a0.y, a0.z, a0.w}, av1[4] = {a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          const float4 wl = *reinterpret_cast<const float4*>(Wcs + (k + kk) * 128 + 4 * tx);
          const float4 wh = *reinterpret_cast<const float4*>(Wcs + (k + kk) * 128 + 64 + 4 * tx);
          const float wv[8] = {wl.x, wl.y, wl.z, wl.w, wh.x, wh.y, wh.z, wh.w};
#pragma unroll
          for (int q = 0; q < 8; ++q) { acc[0][q] = fmaf(av0[kk], wv[q], acc[0][q]); acc[1][q] = fmaf(av1[kk], wv[q], acc[1][q]); }
        }
      }
    }
    // ---- GELU, LayerNorm(128), dot with head.out: per row over its half warp, the same order for every row
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int r = 2 * ty + u;
      int mask = 15, j = 0;
      if (r < 30) { mask = r >> 1; j = min(c * ATTR_CHUNK + (r & 1), M - 1); }
      const float* cs = ((mask & 1) ? pwin : pbg_base + (int64_t)j * ATTR_PROJ) + 4 * 256;
      float hv[8];
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int col = (q < 4 ? 4 * tx + q : 64 + 4 * tx + q - 4);
        hv[q] = attr_gelu(__fadd_rn(__fadd_rn(bcv[q], cs[col]), acc[u][q]));
        s = __fadd_rn(s, hv[q]);
      }
      const float mu = half_warp_sum(s) / 128.0f;
      float d = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) { const float t = __fsub_rn(hv[q], mu); d = __fmaf_rn(t, t, d); }
      const float rstd = 1.0f / sqrtf(half_warp_sum(d) / 128.0f + 1e-5f);
      float o = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) o = __fmaf_rn(__fmaf_rn(__fmul_rn(__fsub_rn(hv[q], mu), rstd), gv[q], bv[q]), wov[q], o);
      o = half_warp_sum(o);
      if (tx == 0) Ls[r] = __fadd_rn(o, bo);
    }
    __syncthreads();
    if (tid < 15) {
      const bool two = c * ATTR_CHUNK + 1 < M;
      partial[((int64_t)i * 15 + tid) * n_chunks + c] = two ? __fadd_rn(Ls[2 * tid], Ls[2 * tid + 1]) : Ls[2 * tid];
    } else if (tid == 15 && c == 0) {
      v15[i] = Ls[30];
    }
  }
}

// One thread per window: v(S) = (sum of the chunks in chunk order) / M for S < 15, v(15) = f(x_i); phi_p = sum over S not
// containing p, in ascending mask order, of w_|S| (v(S | p) - v(S)), w = (1/4, 1/12, 1/12, 1/4).
__global__ void attribution_finalize_kernel(const float* __restrict__ partial, const float* __restrict__ v15, int n, int M,
                                            float* __restrict__ values, float* __restrict__ phi) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int n_chunks = (M + ATTR_CHUNK - 1) / ATTR_CHUNK;
  float v[16];
#pragma unroll
  for (int S = 0; S < 15; ++S) {
    const float* ps = partial + ((int64_t)i * 15 + S) * n_chunks;
    float s = ps[0];
    for (int c = 1; c < n_chunks; ++c) s = __fadd_rn(s, ps[c]);
    v[S] = __fdiv_rn(s, (float)M);
  }
  v[15] = v15[i];
#pragma unroll
  for (int S = 0; S < 16; ++S) values[(int64_t)i * 16 + S] = v[S];
  const float wgt[4] = {1.0f / 4.0f, 1.0f / 12.0f, 1.0f / 12.0f, 1.0f / 4.0f};
#pragma unroll
  for (int p = 0; p < LSD_BRANCHES; ++p) {
    float acc = 0.f;
#pragma unroll
    for (int S = 0; S < 16; ++S) {
      if ((S >> p) & 1) continue;
      const int size = (S & 1) + ((S >> 1) & 1) + ((S >> 2) & 1) + ((S >> 3) & 1);
      acc = __fadd_rn(acc, __fmul_rn(wgt[size], __fsub_rn(v[S | (1 << p)], v[S])));
    }
    phi[(int64_t)i * LSD_BRANCHES + p] = acc;
  }
}

}  // namespace

size_t attribution_tail_smem_bytes() { return (size_t)TAIL_SMEM_FLOATS * sizeof(float); }

cudaError_t attribution_device_init() {
  return cudaFuncSetAttribute(coalition_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attribution_tail_smem_bytes());
}

void launch_branch_attribution(const float* feats, int n, const float* bg, int M, const HeadW& w, float* proj, float* partial,
                               float* v15, float* values, float* phi, int num_sms, cudaStream_t s) {
  const int R = n + M;
  branch_project_kernel<<<(R + PROJ_ROWS - 1) / PROJ_ROWS, 256, 0, s>>>(feats, n, bg, M, w, proj);
  count_launch();
  if (n == 0) return;
  const int64_t n_tiles = (int64_t)n * ((M + ATTR_CHUNK - 1) / ATTR_CHUNK);
  const int grid = (int)std::min<int64_t>(n_tiles, num_sms);
  coalition_tail_kernel<<<grid, TAIL_THREADS, attribution_tail_smem_bytes(), s>>>(proj, n, M, w, partial, v15);
  count_launch();
  attribution_finalize_kernel<<<(n + 127) / 128, 128, 0, s>>>(partial, v15, n, M, values, phi);
  count_launch();
}

}  // namespace lsd
