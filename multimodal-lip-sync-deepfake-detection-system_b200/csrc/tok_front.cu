// Fused front of the token path for sm_100a (see tok_front.cuh): cross-modal attention core + output projections + gated
// fusion + multi-scale Conv1d branches + pre_scale_proj + CLS row, one launch, a CTA per group of windows.
//
// Same machinery as tok_fused.cu: a window owns a slot of SL rows of the 128-row tile (SL >= T + 3, so the Conv1d taps of a
// window read the zero rows that end its slot instead of its neighbour: a window's result does not depend on its slot or on its
// co-tenants, bit for bit); GEMM operands are fp16 planes in shared memory (K-major core matrices, no swizzle), accumulators
// live in TMEM (columns 0..255: the 256-column result being accumulated; 256..511: score / P V / branch tiles), weights stream
// from L2 through a ring of bulk async copies in the order the MMA warp consumes them, compute and MMA phases alternate.
//   * attention: Q / K / V of a head pair come from the in-projection GEMMs (fp32 rows in global memory), are converted to fp16
//     planes (Q scaled by 1/sqrt(32), V transposed), S = Q K^T per window, flash-style un-normalised P, O = P V, and the output
//     projection accumulates over the four head pairs; the next pair's Q / K / V are loaded while the projection runs;
//   * Conv1d over tokens: the A operand of tap j is the fused-token operand with its start address moved by (j - k/2) rows
//     (16 bytes each) — the zero rows behind every window and a zeroed kilobyte in front of the operand supply the padding;
//   * v_out / a_out travel through a small fp32 scratch in global memory (each thread re-reads only what it wrote itself).
#include "tok_front.cuh"

#include "lsd_kernels.h"
#include "tok_common.cuh"
#include "umma.cuh"

namespace lsd {

using namespace umma;
using namespace tokc;

namespace {

constexpr int FR_CWARPS = 16;                        // compute warps: 4 per TMEM lane quarter
constexpr int FR_THREADS = (FR_CWARPS + 2) * 32;     // + weight producer + MMA issuer
constexpr int FR_RING = 5;
constexpr uint32_t OFF_PAD = 0;                      // 1 KB of zeros in front of operand A (rows "before" row 0 for negative Conv1d taps)
constexpr uint32_t OFF_A = 1024;                     // 64 KB: attention output of a head pair (K = 64) / gate input, v half / blend / fused tokens
constexpr uint32_t OFF_B = OFF_A + 65536;            // 80 KB: Q K V^T P during attention; gate input, a half; branch outputs
constexpr uint32_t OFF_QK = OFF_B;                   // Q0 K0 Q1 K1: 4 planes each (hd = 32)
constexpr uint32_t OFF_VT = OFF_QK + 32768;          // V^T of the two heads: [key plane (16)][32 hd rows][8 keys], 8 KB per head
constexpr uint32_t OFF_P = OFF_VT + 16384;           // P of the two heads: <= 8 planes (16 KB) each
constexpr uint32_t P_HEAD = 8 * PLANE;
constexpr uint32_t OFF_RED = OFF_B + 65536;          // partial gate dot products (2 KB), behind the 64 KB operand in region B
constexpr uint32_t OFF_RING = OFF_B + 81920;
constexpr uint32_t FR_SMEM = OFF_RING + FR_RING * TFR_STAGE_BYTES;
static_assert(OFF_P + 2 * P_HEAD <= OFF_RING, "attention buffers must fit in region B");
static_assert(FR_SMEM <= 225 * 1024, "shared-memory budget");
constexpr uint32_t O_COL = 0, ACC_COL = 256;
constexpr int D = 256;

}  // namespace

__global__ void __launch_bounds__(FR_THREADS, 1) tok_front_kernel(const __grid_constant__ TokFrontP p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t w_full[FR_RING], w_empty[FR_RING], bar_mma, bar_cmp;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  constexpr int W_PROD = FR_CWARPS, W_MMA = FR_CWARPS + 1;

  if (tid == 0) {
    for (int i = 0; i < FR_RING; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
    mbar_init(&bar_mma, 1);
    mbar_init(&bar_cmp, FR_CWARPS);
    fence_barrier_init();
  }
  if (tid < 64) st_shared_v4(sbase + OFF_PAD + (uint32_t)tid * 16u, 0u, 0u, 0u, 0u);   // (made visible to the MMAs by these warps' first hand-over)
  if (warp == W_MMA) { tmem_alloc(&tmem_base_s, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const int G = p.G, SL = p.SL, KW = p.KW, T = p.T;

  if (warp == W_PROD) {
    // ------------------------------------------------------------------ weight producer (one lane)
    if (lane == 0) {
      const uint8_t* src = reinterpret_cast<const uint8_t*>(p.w);
      for (int s = 0; s < TFR_N_STAGES; ++s) {
        const int slot = s % FR_RING;
        const uint32_t ph = (uint32_t)(s / FR_RING) & 1u;
        mbar_wait(&w_empty[slot], ph ^ 1u);
        mbar_arrive_expect_tx(&w_full[slot], TFR_STAGE_BYTES);
        bulk_s2(sbase + OFF_RING + (uint32_t)slot * TFR_STAGE_BYTES, src + (size_t)s * TFR_STAGE_BYTES, TFR_STAGE_BYTES, &w_full[slot]);
      }
    }
  } else if (warp == W_MMA) {
    // ------------------------------------------------------------------ MMA issuer (whole warp runs the loop, one lane issues)
    const uint32_t leader = elect_one() ? 1u : 0u;
    const uint64_t desc_hi = ((uint64_t)8 << 32) | ((uint64_t)1 << 46);   // SBO = 128 B, descriptor version 1
    uint32_t par_c = 0;
    int ws = 0;                                                           // weight stages consumed so far
    long long* dbg = (p.dbg && blockIdx.x == 0 && lane == 0) ? reinterpret_cast<long long*>(p.dbg) : nullptr;
    int dbg_n = 0;
    auto wait_cmp = [&]() { mbar_wait(&bar_cmp, par_c); par_c ^= 1u; tc_fence_after(); if (dbg && dbg_n < 64) dbg[2 * dbg_n] = clock64(); };
    auto done = [&]() { mma_commit_pred(&bar_mma, leader); if (dbg && dbg_n < 64) { dbg[2 * dbg_n + 1] = clock64(); ++dbg_n; } };
    auto desc = [&](uint32_t byte_addr, uint32_t lbo_bytes) -> uint64_t {
      return desc_hi | (uint64_t)(((lbo_bytes >> 4) & 0x3FFFu) << 16) | (uint64_t)((byte_addr >> 4) & 0x3FFFu);
    };
    // D[tmem_d] (+)= A[a_addr: planes of 128 rows, K = 16 * k16] * W^T, W = (256 x K) streamed through the ring, 2 K16 steps per stage
    auto gemm_w = [&](uint32_t a_addr, int k16, uint32_t tmem_d, uint32_t acc) {
      const uint32_t idesc = idesc_f16(128, D);
      for (int k0 = 0; k0 < k16; k0 += 2, ++ws) {
        const int slot = ws % FR_RING;
        mbar_wait(&w_full[slot], (uint32_t)(ws / FR_RING) & 1u);
        tc_fence_after();
        const uint32_t wb = sbase + OFF_RING + (uint32_t)slot * TFR_STAGE_BYTES;
#pragma unroll 1
        for (int j = 0; j < 2; ++j) {
          const uint64_t da = desc(a_addr + (uint32_t)(k0 + j) * 2u * PLANE, PLANE);
          const uint64_t db = desc(wb + (uint32_t)j * (uint32_t)D * 32u, (uint32_t)D * 16u);
          mma_bf16_ss_pred(tmem_d, da, db, idesc, acc, leader);
          acc = 1u;
        }
        mma_commit_pred(&w_empty[slot], leader);
      }
    };
    const uint32_t O = tmem + O_COL, ACC = tmem + ACC_COL;
    // S_{h,slot} = Q_h K_{h,slot}^T (see tok_fused.cu): score tile of (h, slot) at ACC + h*128 + slot*SL
    auto mma_scores = [&]() {
      const uint32_t idesc = idesc_f16(128, KW);
#pragma unroll 1
      for (int h = 0; h < 2; ++h)
#pragma unroll 1
        for (int sl = 0; sl < G; ++sl)
#pragma unroll 1
          for (int j = 0; j < 2; ++j) {
            const uint64_t da = desc(sbase + OFF_QK + (uint32_t)(2 * h) * 8192u + (uint32_t)j * 2u * PLANE, PLANE);
            const uint64_t db = desc(sbase + OFF_QK + (uint32_t)(2 * h + 1) * 8192u + (uint32_t)j * 2u * PLANE + (uint32_t)(sl * SL) * 16u, PLANE);
            mma_bf16_ss_pred(ACC + (uint32_t)(h * 128 + sl * SL), da, db, idesc, j ? 1u : 0u, leader);
          }
    };
    // O_{h,slot} = P_h V_{h,slot} at ACC + (h*G + slot)*32
    auto mma_pv = [&]() {
      const uint32_t idesc = idesc_f16(128, 32);
#pragma unroll 1
      for (int h = 0; h < 2; ++h)
#pragma unroll 1
        for (int sl = 0; sl < G; ++sl)
#pragma unroll 1
          for (int j = 0; j < KW / 16; ++j) {
            const uint64_t da = desc(sbase + OFF_P + (uint32_t)h * P_HEAD + (uint32_t)j * 2u * PLANE, PLANE);
            const uint64_t db = desc(sbase + OFF_VT + (uint32_t)h * 8192u + (uint32_t)(sl * SL / 8 + 2 * j) * 512u, 512u);
            mma_bf16_ss_pred(ACC + (uint32_t)((h * G + sl) * 32), da, db, idesc, j ? 1u : 0u, leader);
          }
    };
    // Conv1d branch of kernel size k: tap j reads operand A moved by (j - k/2) rows
    auto branch = [&](int k) {
#pragma unroll 1
      for (int j = 0; j < k; ++j)
        gemm_w((uint32_t)((int)(sbase + OFF_A) + (j - k / 2) * 16), 16, ACC, j ? 1u : 0u);
    };
    for (int dir = 0; dir < 2; ++dir) {
      wait_cmp();                                                         // Q K V of head pair 0
      mma_scores();
      done();
      for (int hp = 0; hp < 4; ++hp) {
        wait_cmp();                                                       // P
        mma_pv();
        done();
        wait_cmp();                                                       // attention output of pair hp (+ Q K V of pair hp+1)
        gemm_w(sbase + OFF_A, 4, O, hp ? 1u : 0u);                        // O (+)= att_hp @ Wo[:, 64hp : 64hp+64]^T
        if (hp < 3) mma_scores();
        done();
      }
    }
    wait_cmp();                                                           // gate input [v_out | a_out]
    gemm_w(sbase + OFF_A, 16, O, 0u);
    gemm_w(sbase + OFF_B, 16, O, 1u);
    done();
    wait_cmp();                                                           // blend
    gemm_w(sbase + OFF_A, 16, O, 0u);
    done();
    wait_cmp();                                                           // fused tokens
    branch(3);
    done();
    wait_cmp();                                                           // GELU'd branch k3
    gemm_w(sbase + OFF_B, 16, O, 0u);
    branch(5);
    done();
    wait_cmp();
    gemm_w(sbase + OFF_B, 16, O, 1u);
    branch(7);
    done();
    wait_cmp();
    gemm_w(sbase + OFF_B, 16, O, 1u);
    done();
  } else {
    // ------------------------------------------------------------------ compute warps: lane quarter q, column quarter cq
    // Two tile-row (= TMEM lane) -> token mappings.  Up to the fused tokens a window's tokens are interleaved over its 4/G lane
    // quarters (token = lane * (4/G) + quarter in window), which spreads the valid rows — and the elementwise work — over all four
    // warp schedulers while a warp's rows still belong to one window (see tok_fused.cu); operands indexed by KEY (K, V^T) are
    // stored in canonical order (krow).  The Conv1d branches need neighbouring tokens in neighbouring operand rows, so the fused
    // tokens are written to canonical rows and everything behind them (branch epilogues, final rows) uses the canonical mapping
    // (window = SL-row slot, token = row in slot).
    const int q = warp & 3, cq = warp >> 2;
    const int row = q * 32 + lane;
    const int QW = 4 / G;
    int slot = q / QW;
    int lrow = lane * QW + (q - slot * QW);
    const int krow = slot * SL + lrow;
    int win = blockIdx.x * G + slot;
    bool valid = slot < G && win < p.B && lrow < T;
    size_t grow = valid ? (size_t)win * T + lrow : 0;                     // row of the (B*T, .) fp32 matrices
    const size_t vgrow = valid ? (size_t)(win / p.K) * T + lrow : 0;      // row of the visual matrices (pv, v_emb)
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    const uint32_t O = lane_base + O_COL, ACC = lane_base + ACC_COL;
    const uint32_t row16 = (uint32_t)row * 16u;
    const int c0 = cq * 64;
    uint32_t par_m = 0;
    long long* dbg = (p.dbg && blockIdx.x == 0 && warp == 0 && lane == 0) ? reinterpret_cast<long long*>(p.dbg) + 128 : nullptr;
    int dbg_n = 0;
    if (dbg) dbg[0] = clock64();
    auto wait_mma = [&]() { mbar_wait(&bar_mma, par_m); par_m ^= 1u; tc_fence_after(); if (dbg && dbg_n < 63) dbg[2 * dbg_n + 2] = clock64(); };
    auto done = [&]() {
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_cmp);
      if (dbg && dbg_n < 63) { dbg[2 * dbg_n + 1] = clock64(); ++dbg_n; }
    };
    auto quarter_sync = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(2 + q) : "memory"); };   // the four warps of this lane quarter
    // 32 consecutive fp32 of a global row (zeros for rows outside the batch)
    auto ld_row32 = [&](const float* src, float* v) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float4 t = valid ? __ldg(reinterpret_cast<const float4*>(src) + e) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[4 * e] = t.x; v[4 * e + 1] = t.y; v[4 * e + 2] = t.z; v[4 * e + 3] = t.w;
      }
    };
    auto ld_row32_nc = [&](const float* src, float* v) {                   // same, for scratch this kernel wrote (no read-only path)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float4 t = valid ? *(reinterpret_cast<const float4*>(src) + e) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[4 * e] = t.x; v[4 * e + 1] = t.y; v[4 * e + 2] = t.z; v[4 * e + 3] = t.w;
      }
    };
    auto st_row32 = [&](float* dst, const float* v) {
#pragma unroll
      for (int e = 0; e < 8; ++e) *(reinterpret_cast<float4*>(dst) + e) = make_float4(v[4 * e], v[4 * e + 1], v[4 * e + 2], v[4 * e + 3]);
    };
    auto st_planes32 = [&](uint32_t base, const float* v) {                // 32 columns -> 4 planes
#pragma unroll
      for (int j = 0; j < 4; ++j) st_plane8(base + (uint32_t)j * PLANE + row16, v + 8 * j);
    };
    // Q K V of head pair hp of direction dir -> fp16 planes.  dir 0 (v2a): Q from the visual tokens, K / V from the audio tokens;
    // dir 1 (a2v): the other way round.  cq 0: Q0 K0, cq 1: Q1 K1, cq 2: V0, cq 3: V1 (the transposing stores alone).
    auto load_qkv = [&](int dir, int hp) {
      const float* qsrc = dir == 0 ? p.pv + vgrow * p.ld_p : p.pa + grow * p.ld_p;
      const float* kvsrc = dir == 0 ? p.pa + grow * p.ld_p : p.pv + vgrow * p.ld_p;
      float v[32];
      if (cq < 2) {
        const int head = 2 * hp + cq;
        ld_row32(qsrc + head * 32, v);
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] *= 0.17677669529663688f;
        st_planes32(sbase + OFF_QK + (uint32_t)(2 * cq) * 8192u, v);
        ld_row32(kvsrc + 256 + head * 32, v);
#pragma unroll
        for (int j = 0; j < 4; ++j) st_plane8(sbase + OFF_QK + (uint32_t)(2 * cq + 1) * 8192u + (uint32_t)j * PLANE + (uint32_t)krow * 16u, v + 8 * j);
      } else {
        const int h = cq - 2, head = 2 * hp + h;
        ld_row32(kvsrc + 512 + head * 32, v);
        const uint32_t base = sbase + OFF_VT + (uint32_t)h * 8192u + (uint32_t)(krow >> 3) * 512u + (uint32_t)(krow & 7) * 2u;
#pragma unroll
        for (int d = 0; d < 32; ++d) st_shared_u16(base + (uint32_t)d * 16u, __half_as_ushort(__float2half_rn(v[d])));
      }
    };
    const float* vec = p.vec;
    float inv_sum = 0.f;

    load_qkv(0, 0);
    done();
    for (int dir = 0; dir < 2; ++dir) {
      for (int hp = 0; hp < 4; ++hp) {
        // ---- softmax over the row's own window (score columns slot*SL .. +T of head cq), un-normalised P -> fp16 planes
        wait_mma();
        if (cq < 2) {
          const uint32_t S = ACC + (uint32_t)(cq * 128 + slot * SL);
          float mx = -INFINITY;
#pragma unroll 1
          for (int k0 = 0; k0 < T; k0 += 32) {
            float v[32];
            tmem_ld32(S + (uint32_t)k0, v);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) if (k0 + e < T) mx = fmaxf(mx, v[e]);
          }
          float sum = 0.f;
          const uint32_t pbase = sbase + OFF_P + (uint32_t)cq * P_HEAD + row16;
#pragma unroll 1
          for (int k0 = 0; k0 < KW; k0 += 32) {
            float v[32];
            tmem_ld32(S + (uint32_t)k0, v);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              const float pe = (valid && k0 + e < T) ? __expf(v[e] - mx) : 0.f;
              const float pr = __half2float(__float2half_rn(pe));        // the row sum is taken over what the tensor core multiplies with V
              sum += pr;
              v[e] = pr;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (k0 + 8 * j < KW) st_plane8(pbase + (uint32_t)(k0 / 8 + j) * PLANE, v + 8 * j);
          }
          inv_sum = (valid && sum > 0.f) ? 1.0f / sum : 0.f;
        }
        done();
        // ---- attention output of head 2hp + cq -> planes 4cq..4cq+3 of the K = 64 operand; next pair's Q K V
        wait_mma();
        if (cq < 2) {
          float v[32];
          tmem_ld32(ACC + (uint32_t)((cq * G + slot) * 32), v);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] *= inv_sum;
          st_planes32(sbase + OFF_A + (uint32_t)(4 * cq) * PLANE, v);
        }
        if (hp < 3) load_qkv(dir, hp + 1);
        done();
      }
      // ---- out = O + bias + residual -> scratch [v_out | a_out]; then the next direction's first Q K V, or the gate input planes
      wait_mma();
      {
        const float* res = dir == 0 ? p.v_emb + vgrow * p.ld_e : p.a_int + grow * p.ld_e;
        const float* bo = vec + (dir == 0 ? TFR_V_BO0 : TFR_V_BO1);
        float* dst = p.gi + grow * 512 + dir * D;
#pragma unroll 1
        for (int c = c0; c < c0 + 64; c += 32) {
          float v[32], r[32];
          tmem_ld32(O + (uint32_t)c, v);
          tmem_ld_wait();
          add32(v, bo + c);
          ld_row32(res + c, r);
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = valid ? v[e] + r[e] : 0.f;
          if (valid) st_row32(dst + c, v);
          if (dir == 1) st_planes32(sbase + OFF_B + (uint32_t)(c / 8) * PLANE, v);   // a half of the gate input (K chunks 16..31)
        }
      }
      if (dir == 0) {
        load_qkv(1, 0);
      } else {
#pragma unroll 1
        for (int c = c0; c < c0 + 64; c += 32) {                          // v half of the gate input
          float v[32];
          ld_row32_nc(p.gi + grow * 512 + c, v);
          st_planes32(sbase + OFF_A + (uint32_t)(c / 8) * PLANE, v);
        }
      }
      done();
    }
    // ---- gate: g = sigmoid(GELU(O + b0) . w2 + b2);  blend = g * v_out + (1 - g) * a_out   (fusion_module.py:84-86)
    wait_mma();
    {
      float dot = 0.f;
#pragma unroll 1
      for (int c = c0; c < c0 + 64; c += 32) {
        float v[32];
        tmem_ld32(O + (uint32_t)c, v);
        tmem_ld_wait();
        add32(v, vec + TFR_V_BG0 + c);
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(vec + TFR_V_WG2 + c) + e4);
          dot = fmaf(gelu_fast(v[4 * e4]), w.x, dot);
          dot = fmaf(gelu_fast(v[4 * e4 + 1]), w.y, dot);
          dot = fmaf(gelu_fast(v[4 * e4 + 2]), w.z, dot);
          dot = fmaf(gelu_fast(v[4 * e4 + 3]), w.w, dot);
        }
      }
      const uint32_t red = sbase + OFF_RED + (uint32_t)row * 4u;           // [4 cq][128 rows] floats
      st_shared_f32(red + (uint32_t)cq * 512u, dot);
      quarter_sync();
      const float z = ((ld_shared_f32(red) + ld_shared_f32(red + 512u)) + (ld_shared_f32(red + 1024u) + ld_shared_f32(red + 1536u))) + __ldg(vec + TFR_V_BG2);
      const float g = 1.0f / (1.0f + expf(-z));
#pragma unroll 1
      for (int c = c0; c < c0 + 64; c += 32) {
        float a[32], b[32];
        ld_row32_nc(p.gi + grow * 512 + c, a);
        ld_row32_nc(p.gi + grow * 512 + D + c, b);
#pragma unroll
        for (int e = 0; e < 32; ++e) a[e] = valid ? g * a[e] + (1.0f - g) * b[e] : 0.f;
        st_planes32(sbase + OFF_A + (uint32_t)(c / 8) * PLANE, a);
      }
    }
    done();
    // ---- fused = ReLU(O + b)  (fusion_module.py:87) -> fp32 rows + operand A of the Conv1d branches (zero rows outside the window)
    wait_mma();
#pragma unroll 1
    for (int c = c0; c < c0 + 64; c += 32) {
      float v[32];
      tmem_ld32(O + (uint32_t)c, v);
      tmem_ld_wait();
      add32(v, vec + TFR_V_BF + c);
#pragma unroll
      for (int e = 0; e < 32; ++e) v[e] = valid ? fmaxf(v[e], 0.f) : 0.f;
      if (valid) st_row32(p.fused + grow * D + c, v);
#pragma unroll
      for (int j = 0; j < 4; ++j) st_plane8(sbase + OFF_A + (uint32_t)(c / 8 + j) * PLANE + (uint32_t)krow * 16u, v + 8 * j);   // canonical row
    }
    __threadfence_block();             // the fused rows are re-read below by the thread that owns the token in the canonical mapping
    done();
    // ---- canonical mapping from here on
    slot = (q * 32) / SL;
    lrow = row - slot * SL;
    win = blockIdx.x * G + slot;
    valid = slot < G && win < p.B && lrow < T;
    grow = valid ? (size_t)win * T + lrow : 0;
    // ---- branches: GELU(acc + BN shift) -> operand of the pre_scale_proj slice  (temporal.py:95-103)
#pragma unroll 1
    for (int b = 0; b < 3; ++b) {
      wait_mma();
      const float* sh = vec + (b == 0 ? TFR_V_SH3 : (b == 1 ? TFR_V_SH5 : TFR_V_SH7));
#pragma unroll 1
      for (int c = c0; c < c0 + 64; c += 32) {
        float v[32];
        tmem_ld32(ACC + (uint32_t)c, v);
        tmem_ld_wait();
        add32(v, sh + c);
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = valid ? gelu_fast(v[e]) : 0.f;
        st_planes32(sbase + OFF_B + (uint32_t)(c / 8) * PLANE, v);
      }
      done();
    }
    // ---- tok rows 1..T = fused + pre_scale_proj(cat) + bias; row 0 = cls token  (temporal.py:104-107)
    wait_mma();
    if (__any_sync(0xffffffffu, valid)) {                                  // warp-uniform: tcgen05.ld is .sync.aligned
      float* trow = p.tok + ((size_t)(valid ? win : 0) * (T + 1) + 1 + (valid ? lrow : 0)) * D;
#pragma unroll 1
      for (int c = c0; c < c0 + 64; c += 32) {
        float v[32], f[32];
        tmem_ld32(O + (uint32_t)c, v);
        tmem_ld_wait();
        add32(v, vec + TFR_V_BP + c);
        ld_row32_nc(p.fused + grow * D + c, f);
        if (valid) {
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] += f[e];
          st_row32(trow + c, v);
          if (lrow == 0) {
            float cl[32];
            ld_row32(vec + TFR_V_CLS + c, cl);
            st_row32(trow - D + c, cl);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tmem_dealloc(tmem, 512);
}

cudaError_t tok_front_device_init() {
  return cudaFuncSetAttribute(tok_front_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FR_SMEM);
}

// Row slot per window: a multiple of 32 (a warp's rows belong to one window) with at least 3 zero rows behind the window's T
// tokens (the k = 7 branch reaches 3 rows past either end).  KW = key extent per window (multiple of 16).
void tok_front_geometry(int T, int& SL, int& G, int& KW) {
  SL = T + 3 <= 32 ? 32 : 64;
  G = 128 / SL;
  KW = (T + 15) / 16 * 16;
}
bool tok_front_supported(int T) { return T >= 1 && T + 3 <= 64; }

void launch_tok_front(const TokFrontP& p, cudaStream_t s) {
  const int grid = (p.B + p.G - 1) / p.G;
  if (grid <= 0) return;
  tok_front_kernel<<<grid, FR_THREADS, FR_SMEM, s>>>(p);
  count_launch();
}

}  // namespace lsd
