// "Temporal ring" stem convolution for sm_100a: Conv3d(3 -> 64, kernel (3,7,7), stride (1,2,2), pad (1,3,3)) + eval BatchNorm + ReLU
// (app/models/visual_encoder.py:113-125) on tcgen05, with the three temporal taps folded into the N dimension of the MMA.
//
// Why: a 64-column MMA (M = 128, K = 16) reads 4 KB of A and 2 KB of B from shared memory for 32 cycles of tensor work — the 128 B/cycle
// read port, not the tensor pipe, paces it (48 cycles).  The A operand of the three temporal taps of one input slab is the SAME shared-
// memory view; only the weights differ.  So one MMA with B = [W(dt=-1) | W(dt=0) | W(dt=+1)] (N = 192) reads A once for three times the
// FLOPs (4 + 6 KB = 80 cycles of port for 96 cycles of tensor work: tensor-bound), and its three 64-column blocks are the contributions
// of input slab t to the outputs t+1, t, t-1.  An accumulator slot therefore walks ONE 128-position column chunk along t and keeps a
// ring of four 64-column blocks in TMEM: at step t the MMAs add into [out(t+1) | out(t) | out(t-1)], out(t-1) is then complete and
// is drained by the epilogue while step t+1 runs, and the block that held out(t-2) restarts as out(t+2) (initialised to the bias by
// one extra MMA, like the lean epilogue of umma_conv.cu).  The D region moves down by one block per step; where it would wrap around the
// ring it is issued as two MMAs (N = 128 + 64).
//
// Work split: the (column chunk, t) outputs are numbered column-major and cut into equal contiguous ranges, one per accumulator slot
// (two slots per CTA, 512 TMEM columns); a range that starts or ends inside a column pays one halo step per cut (the host expands the
// ranges into a step table, SrStep).  The 84 KB of weights stay resident in shared memory for the whole kernel; per step only the two
// pixel-row regions of the chunk (Toeplitz K: rows and K chunks are 16-byte shifts of one region, see umma_conv.cuh) are streamed in.
// The summation order of an output (bias, then slabs t-1, t, t+1, each over parity sets, rows and K chunks) does not depend on how
// the ranges are cut, so logits stay independent of the batch composition bit for bit.
//
// Warp roles (384 threads): warp 0 producer, warps 1-2 MMA issuers (one per slot), warp 3 TMEM allocation, warps 4-11 epilogue
// (warps 4-7 slot 0, 8-11 slot 1; warp % 4 = TMEM lane quarter).
#include "stem_ring.cuh"

#include <cstdio>

#include "lsd_kernels.h"
#include "umma.cuh"

namespace lsd {

using namespace umma;

namespace {

constexpr int SR_NST = 6;   // SR_NST: most ring stages (barrier arrays); p.nst are in use
constexpr int SR_THREADS = 384;

__device__ __forceinline__ uint32_t sr_div(uint32_t n, uint32_t m, int s) { return (uint32_t)(((uint64_t)n * m) >> (31 + s)); }
__device__ __forceinline__ bool sr_valid(const UcGeom& g, int64_t P) {
  if (P < 0 || P >= g.P_total) return false;
  const uint32_t Pu = (uint32_t)P;
  const uint32_t S = sr_div(Pu, g.mSL, g.sSL);
  const int r = (int)(Pu - S * (uint32_t)g.SL);
  const int row = (int)sr_div((uint32_t)r, g.mRW, g.sRW), col = r - row * g.RW;
  const int n = (int)sr_div(S, g.mTS, g.sTS);
  const int t = (int)(S - (uint32_t)n * (uint32_t)g.TS) - g.ot;
  const int h = row - g.oh, w = col - g.ow;
  return (unsigned)t < (unsigned)g.T && (unsigned)h < (unsigned)g.H && (unsigned)w < (unsigned)g.W && n < g.N;
}
__device__ __forceinline__ uint4 sr_pack8_relu(const float* v) {
  uint4 o;
  uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
  for (int e = 0; e < 4; ++e) asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(ow[e]) : "f"(v[2 * e + 1]), "f"(v[2 * e]));
  return o;
}

__global__ void __launch_bounds__(SR_THREADS, 1) stem_ring_kernel(const __grid_constant__ StemRingP p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t full_bar[SR_NST], empty_bar[SR_NST], tfull[2][4], tempty[2][4], wbar;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t r0 = ((uint32_t)p.units[0] * 16u + 127u) & ~127u, r1 = ((uint32_t)p.units[1] * 16u + 127u) & ~127u;
  const uint32_t slot_bytes = r0 + r1, stage_bytes = 2u * slot_bytes;
  uint8_t* const wsm = smem;                       // resident weights
  uint8_t* const ones = smem + SR_WBYTES;          // A of the bias MMA: 128 rows x (1, 1, 1, 0, ...), both K halves alias it (LBO = 0)
  uint8_t* const biasb = ones + 2048;              // B of the bias MMA: [2 K halves][64 columns][8]: (hi, mid, lo) parts of the bias, zeros
  uint8_t* const stages = biasb + 2048;
  // this CTA's two rows of the step table, behind the stages (a dependent global load per step in every role's loop cost ~700 cycles
  // of L2 latency per step on the critical path)
  SrStep* const tab = reinterpret_cast<SrStep*>(stages + (size_t)p.nst * stage_bytes);

  {
    const uint2* src = reinterpret_cast<const uint2*>(p.steps + (size_t)(2 * blockIdx.x) * (size_t)p.nsteps);
    for (int i = tid; i < 2 * p.nsteps; i += SR_THREADS) reinterpret_cast<uint2*>(tab)[i] = src[i];
  }
  if (tid == 0) {
    for (int i = 0; i < SR_NST; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 2); }
    for (int s = 0; s < 2; ++s)
      for (int i = 0; i < 4; ++i) { mbar_init(&tfull[s][i], 1); mbar_init(&tempty[s][i], 4); }
    mbar_init(&wbar, 1);
    fence_barrier_init();
  }
  if (warp == 3) { tmem_alloc(&tmem_base_s, 512); tmem_relinquish(); }
  if (tid < 128) {
    reinterpret_cast<uint4*>(ones)[tid] = make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u);
    uint4 o = make_uint4(0u, 0u, 0u, 0u);
    if (tid < 64 && p.bias) {
      const float b = p.bias[tid];
      const __nv_bfloat16 hi = __float2bfloat16_rn(b);
      const float e1 = b - __bfloat162float(hi);
      const __nv_bfloat16 mid = __float2bfloat16_rn(e1);
      const __nv_bfloat16 lo = __float2bfloat16_rn(e1 - __bfloat162float(mid));
      o.x = (uint32_t)__bfloat16_as_ushort(hi) | ((uint32_t)__bfloat16_as_ushort(mid) << 16);
      o.y = (uint32_t)__bfloat16_as_ushort(lo);
    }
    reinterpret_cast<uint4*>(biasb)[tid] = o;
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const SrStep* const st0 = tab;
  long long* const dbg = (p.dbg && blockIdx.x == 0 && lane == 0) ? p.dbg : nullptr;
  // (per-CTA span: [256 + 4*cta + {0: globaltimer at start, 1: at end, 2: clock64 at start, 3: at end}])
  unsigned long long gt0 = 0;
  long long ck0 = 0;
  if (p.dbg && tid == 0) { asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt0)); ck0 = clock64(); }
  auto stamp = [&](int role, int k, int which) { if (dbg && k >= 16 && k < 48) dbg[(role * 32 + (k - 16)) * 2 + which] = clock64(); };

  if (warp == 0) {
    // ------------------------------------------------ producer: the weights once, then per step the pixel-row regions of both slots
    if (lane == 0) {
      mbar_arrive_expect_tx(&wbar, (uint32_t)SR_WBYTES);
      bulk_g2s(wsm, p.w, (uint32_t)SR_WBYTES, &wbar);
    }
    const int slot = (lane >> 1) & 1, set = lane & 1;
    const SrStep* const st = st0 + (size_t)slot * (size_t)p.nsteps;
    const uint32_t bytes = (uint32_t)p.units[set] * 16u;
    const uint32_t dst0 = smem_u32(stages) + (uint32_t)slot * slot_bytes + (set ? r0 : 0u);
    for (int k = 0; k < p.nsteps; ++k) {
      const int stage = k % p.nst;
      const uint32_t ph = (uint32_t)(k / p.nst) & 1u;
      const SrStep sd = st[k];
      const bool act = lane < 4 && (sd.flags & SR_ACTIVE);
      const uint32_t total = __reduce_add_sync(0xffffffffu, act ? bytes : 0u);
      mbar_wait(&empty_bar[stage], ph ^ 1u);
      stamp(0, k, 0);
      if (lane == 0) mbar_arrive_expect_tx(&full_bar[stage], total);
      __syncwarp();
      if (act) {
        const __nv_bfloat16* src = p.xs[set] + ((int64_t)sd.in_pos + (int64_t)p.start[set]) * 8;
        bulk_s2(dst0 + (uint32_t)stage * stage_bytes, src, bytes, &full_bar[stage]);
      }
      __syncwarp();
      stamp(0, k, 1);
    }
  } else if (warp == 1 || warp == 2) {
    // ------------------------------------------------ MMA issuer of slot (warp - 1): whole warp runs the loop, one lane issues
    const int slot = __shfl_sync(0xffffffffu, warp, 0) - 1;
    const SrStep* const st = st0 + (size_t)slot * (size_t)p.nsteps;
    const uint32_t leader = elect_one() ? 1u : 0u;
    const uint64_t desc_hi64 = ((uint64_t)8 << 32) | ((uint64_t)1 << 46);          // SBO = 128 B, descriptor version 1
    const uint32_t id192 = (p.skip & 8) ? idesc_bf16(128, 64) : idesc_bf16(128, 192), id128 = idesc_bf16(128, 128), id64 = idesc_bf16(128, 64);   // (skip bit 3: timing experiment)
    const uint32_t tb = tmem + (uint32_t)slot * 256u;
    const uint64_t d_ones = desc_hi64 | (uint64_t)(smem_u32(ones) >> 4);                           // LBO = 0
    const uint64_t d_bias = desc_hi64 | (uint64_t)((smem_u32(biasb) >> 4) | (64u << 16));         // LBO = 64 columns x 16 B
    const uint32_t w0 = (smem_u32(wsm) >> 4) | (192u << 16);                                       // LBO = 192 columns x 16 B
    const uint32_t a_slot = (smem_u32(stages) + (uint32_t)slot * slot_bytes) >> 4;
    mbar_wait(&wbar, 0u);
    tc_fence_after();
    int q = 0;
    for (int k = 0; k < p.nsteps; ++k) {
      const int stage = k % p.nst;
      const uint32_t ph = (uint32_t)(k / p.nst) & 1u;
      // (a value ptxas knows to be warp-uniform: everything derived from it — q, the D block, the branches — then stays in uniform
      //  registers; taken straight from the shared-memory load, every MMA operand went through R2UR moves, ~4 per MMA)
      const uint32_t flags = __shfl_sync(0xffffffffu, st[k].flags, 0);
      mbar_wait(&full_bar[stage], ph);
      tc_fence_after();
      if (slot == 0) stamp(1, k, 0);
      if (flags & SR_ACTIVE) {
        if (q >= 2) { mbar_wait(&tempty[slot][(q - 2) & 3], (uint32_t)((q - 2) >> 2) & 1u); tc_fence_after(); }
        if (slot == 0) stamp(1, k, 1);
        const uint32_t c = (p.skip & 2) ? 0u : ((uint32_t)(-q) & 3u);   // first block of this step's D region: [out(t+1) | out(t) | out(t-1)]
        if (flags & SR_FIRST) {
          mma_bf16_ss_pred(tb + c * 64u, d_ones, d_bias, id64, 0u, leader);
          mma_bf16_ss_pred(tb + ((c + 1u) & 3u) * 64u, d_ones, d_bias, id64, 0u, leader);
          mma_bf16_ss_pred(tb + ((c + 2u) & 3u) * 64u, d_ones, d_bias, id64, 0u, leader);
        } else {
          mma_bf16_ss_pred(tb + c * 64u, d_ones, d_bias, id64, 0u, leader);
        }
        // (descriptors advance by running additions — taps of a parity set are RW positions apart, weight blocks are consecutive — so
        //  the loop carries no loads and few live uniform registers; an unrolled version with per-tap offsets kept in an array went
        //  through vector registers and R2UR moves, ~4 per MMA)
        const uint32_t ab = a_slot + (((uint32_t)stage * stage_bytes) >> 4) + (1u << 16);   // LBO = 16 B (Toeplitz K)
        const uint32_t rw = (uint32_t)p.g.RW;
        uint32_t wj = w0;
#pragma unroll 1
        for (int set = 0; set < 2; ++set) {
          uint32_t at = ab + (set ? (r0 >> 4) : 0u);
          const int nt = set ? 4 : 3;
#pragma unroll 1
          for (int tp = 0; tp < nt; ++tp, at += rw, wj += 2u * (uint32_t)(SR_WBLOCK >> 4)) {
            if ((p.skip & 4) && (set || tp >= 2)) continue;
            const uint64_t da0 = desc_hi64 | (uint64_t)at, da1 = desc_hi64 | (uint64_t)(at + 2u);
            const uint64_t db0 = desc_hi64 | (uint64_t)wj, db1 = desc_hi64 | (uint64_t)(wj + (uint32_t)(SR_WBLOCK >> 4));
            if (c <= 1u) {
              mma_bf16_ss_pred(tb + c * 64u, da0, db0, id192, 1u, leader);
              mma_bf16_ss_pred(tb + c * 64u, da1, db1, id192, 1u, leader);
            } else if (c == 2u) {          // blocks 2, 3, then (wrapped) block 0
              mma_bf16_ss_pred(tb + 128u, da0, db0, id128, 1u, leader);
              mma_bf16_ss_pred(tb, da0, db0 + 128u, id64, 1u, leader);
              mma_bf16_ss_pred(tb + 128u, da1, db1, id128, 1u, leader);
              mma_bf16_ss_pred(tb, da1, db1 + 128u, id64, 1u, leader);
            } else {                       // block 3, then (wrapped) blocks 0, 1
              mma_bf16_ss_pred(tb + 192u, da0, db0, id64, 1u, leader);
              mma_bf16_ss_pred(tb, da0, db0 + 64u, id128, 1u, leader);
              mma_bf16_ss_pred(tb + 192u, da1, db1, id64, 1u, leader);
              mma_bf16_ss_pred(tb, da1, db1 + 64u, id128, 1u, leader);
            }
          }
        }
        mma_commit_pred(&tfull[slot][q & 3], leader);   // out(t-1) of this slot is complete
        if (slot == 0) stamp(2, k, 0);
        ++q;
      }
      mma_commit_pred(&empty_bar[stage], leader);       // the stage is free once the MMAs that read it have completed
    }
  } else if (warp >= 4) {
    // ------------------------------------------------ epilogue: drain the completed block (thread = position), ReLU, bf16, planar store
    const int slot = (warp - 4) >> 2, quarter = warp & 3;
    const SrStep* const st = st0 + (size_t)slot * (size_t)p.nsteps;
    const int i = quarter * 32 + lane;
    int q = 0;
    for (int k = 0; k < p.nsteps; ++k) {
      const SrStep sd = st[k];
      if (!(sd.flags & SR_ACTIVE)) continue;
      mbar_wait(&tfull[slot][q & 3], (uint32_t)(q >> 2) & 1u);
      tc_fence_after();
      if (warp == 4) stamp(3, k, 0);
      if ((sd.flags & SR_STORE) && !(p.skip & 1)) {
        const uint32_t blk = (((uint32_t)(-q) & 3u) + 2u) & 3u;
        const uint32_t ta = tmem + (uint32_t)slot * 256u + blk * 64u + ((uint32_t)(quarter * 32) << 16);
        const bool store = i < (int)((sd.flags >> 8) & 0xffu);
        const int64_t P = (int64_t)sd.in_pos - p.g.SL + i;
        const uint32_t vmask = (store && sr_valid(p.g, P)) ? 0xffffffffu : 0u;     // pad positions of the slab are written as zeros
        char* yp = reinterpret_cast<char*>(p.y + P * 8);
        const int64_t yps = p.y_plane_stride * 2;
#pragma unroll 1
        for (int c0 = 0; c0 < 64; c0 += 32, yp += 4 * yps) {
          float v[32];
          tmem_ld32(ta + (uint32_t)c0, v);
          tmem_ld_wait();
          if (store) {
#pragma unroll
            for (int qq = 0; qq < 4; ++qq) {
              uint4 o = sr_pack8_relu(v + 8 * qq);
              o.x &= vmask; o.y &= vmask; o.z &= vmask; o.w &= vmask;
              *reinterpret_cast<uint4*>(yp + qq * yps) = o;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[slot][q & 3]);
      if (warp == 4) stamp(3, k, 1);
      ++q;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (p.dbg && tid == 0 && blockIdx.x < 160) {
    unsigned long long gt1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1));
    long long* d = p.dbg + 256 + 4 * blockIdx.x;
    d[0] = (long long)gt0; d[1] = (long long)gt1; d[2] = ck0; d[3] = clock64();
  }
  if (warp == 3) tmem_dealloc(tmem, 512);
}

}  // namespace

size_t stem_ring_smem_bytes(const StemRingP& p) {
  const size_t r0 = ((size_t)p.units[0] * 16 + 127) & ~size_t(127), r1 = ((size_t)p.units[1] * 16 + 127) & ~size_t(127);
  return (size_t)SR_WBYTES + 4096 + (size_t)p.nst * 2 * (r0 + r1) + (size_t)2 * p.nsteps * sizeof(SrStep) + 1024;
}

cudaError_t stem_ring_device_init() {
  return cudaFuncSetAttribute(stem_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 223 * 1024);
}

void launch_stem_ring(const StemRingP& p, int grid, cudaStream_t s) {
  if (grid <= 0 || p.nsteps <= 0) return;
  stem_ring_kernel<<<grid, SR_THREADS, stem_ring_smem_bytes(p), s>>>(p);
  count_launch();
}

}  // namespace lsd
