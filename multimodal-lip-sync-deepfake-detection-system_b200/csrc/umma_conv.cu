// tcgen05 "flat shift-GEMM" convolution for sm_100a (bf16 operands, fp32 accumulation in TMEM).
//
// Replaces nn.Conv3d / Conv2d / Conv1d / Linear + eval BatchNorm + ReLU/GELU + residual of the reference
// (app/models/visual_encoder.py:46-87, audio_encoder.py:34-89, artifact_detector.py:74-93,41-43, temporal.py:35-51)
// on the bf16 path.  See umma_conv.cuh for the padded planar activation layout that turns every tap into a shift.
//
// One CTA = MT consecutive 128-position M tiles x all Cout (<= 256) columns; accumulators in TMEM (MT*Cout columns).
// Pipeline (mbarrier ring, `stages` deep), per (k16 channel chunk, band):
//   producer thread : 3 bulk async copies (TMA engine, 1-D): the band's two 8-channel planes + the band's packed weights
//   MMA thread      : ntaps x MT tcgen05.mma (M=128, N=Cout, K=16); the A descriptor of a tap is the band base shifted by the
//                     tap offset (K-major, SWIZZLE_NONE: rows 16 B apart, SBO = 128 B, LBO = band length * 16 B)
//   tcgen05.commit releases the stage; the last commit signals the epilogue.
// Epilogue (all 4 warps): tcgen05.ld -> +bias (+residual) -> act -> zero pads -> bf16 -> 16 B coalesced stores per plane.
#include "umma_conv.cuh"
#include "token_kernels.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "lsd_kernels.h"
#include "umma.cuh"

namespace lsd {

using namespace umma;

struct F8 { float v[8]; };
// exact (erf) GELU of 8 values, kept out of line (register ABI) so that the unrolled epilogue step holds one copy of erff
__device__ __noinline__ F8 gelu8(F8 x) {
#pragma unroll
  for (int e = 0; e < 8; ++e) x.v[e] = 0.5f * x.v[e] * (1.0f + erff(x.v[e] * 0.70710678118654752f));
  return x;
}

__device__ __forceinline__ float uc_act(float v, int act) {
  if (act == ACT_RELU) return fmaxf(v, 0.0f);
  if (act == ACT_GELU) return 0.5f * v * (1.0f + erff(v * 0.70710678118654752f));
  return v;
}

// (P_total < 2^31 is enforced on the host: the three divisions are multiply + shift with the geometry's magic numbers)
__device__ __forceinline__ uint32_t uc_div(uint32_t n, uint32_t m, int s) { return (uint32_t)(((uint64_t)n * m) >> (31 + s)); }
__device__ __forceinline__ bool uc_decode(const UcGeom& g, int64_t P, int& n, int& t, int& h, int& w) {
  if (P < 0 || P >= g.P_total) return false;
  const uint32_t Pu = (uint32_t)P;
  const uint32_t S = uc_div(Pu, g.mSL, g.sSL);
  const int r = (int)(Pu - S * (uint32_t)g.SL);
  const int row = (int)uc_div((uint32_t)r, g.mRW, g.sRW), col = r - row * g.RW;
  n = (int)uc_div(S, g.mTS, g.sTS);
  t = (int)(S - (uint32_t)n * (uint32_t)g.TS) - g.ot;
  h = row - g.oh; w = col - g.ow;
  return (unsigned)t < (unsigned)g.T && (unsigned)h < (unsigned)g.H && (unsigned)w < (unsigned)g.W && n < g.N;
}

__device__ __forceinline__ int64_t uc_flat(const UcGeom& g, int n, int t, int h, int w) {
  return (((int64_t)n * g.TS + t + g.ot) * g.HP + h + g.oh) * g.RW + w + g.ow;
}

__device__ __forceinline__ uint4 pack8(const float* v) {
  uint4 o;
  __nv_bfloat162* ob = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
  for (int e = 0; e < 4; ++e) ob[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
  return o;
}
// same with the ReLU folded into the conversion (cvt.rn.relu.bf16x2.f32: negative inputs and -0 give +0)
__device__ __forceinline__ uint4 pack8_relu(const float* v) {
  uint4 o;
  uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
  for (int e = 0; e < 4; ++e) asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(ow[e]) : "f"(v[2 * e + 1]), "f"(v[2 * e]));
  return o;
}
__device__ __forceinline__ void unpack8(const uint4& r, float* v) {
  const __nv_bfloat162* rb = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
  for (int e = 0; e < 4; ++e) { const float2 f = __bfloat1622float2(rb[e]); v[2 * e] = f.x; v[2 * e + 1] = f.y; }
}

// Persistent, warp-specialised (16 warps):
//   warps 0-3  bulk-copy producers: ring stage k of the CTA's stream belongs to warp k % 4, whose lanes issue the stage's
//              copies (2 planes per K chunk + the weight pieces) in one converged cp.async.bulk; operands come from the
//              stage program in shared memory (see UcStageDesc in umma_conv.cuh),
//   warps 4-7  MMA issuers (1, 2 or 4 active; each owns an equal share of the tile's M-tiles); the loop nest runs
//              warp-uniformly, only the tcgen05.mma / tcgen05.commit are predicated on one elected lane,
//   warps 8-15 epilogue (two warps per TMEM lane quarter, each handling half of the columns).
// Tile walk (static stride): each CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ... of its column slice (a folded conv
// launches one CTA per tile).  On CTA pairs (MODE 3) the walk runs over tile pairs instead: pair blockIdx.x / 2 takes pairs
// j, j + gridDim.x / 2, ..., and each CTA of a pair computes tile 2j + its rank in the cluster.  The accumulators are
// double-buffered in TMEM when they fit so that the epilogue of tile i overlaps the main loop of tile i+1, and the smem ring keeps
// streaming across tile boundaries.
constexpr int UC_THREADS = 512;
constexpr int UC_PROD_WARPS = 4, UC_MMA_WARP0 = 4, UC_MMA_WARPS = 4, UC_EPI_WARP0 = 8, UC_EPI_WARPS = 8;
// (issuing one cp.async.bulk occupies the issuing thread for ~330 cycles; the cost overlaps across warps and partly across the
// lanes of a warp — probe/bulk_issue.cu — hence one stage per warp and one copy per lane; a stage has at most 3 * kpack <= 24
// copies, checked on the host)

// GENERIC = false: lean epilogue of the convolution layers (bias, ReLU/none, optional bf16 residual, planar / parity-split bf16
// store).  GENERIC = true: everything (fp32 rows in/out, split-bf16 hi/lo outputs and residuals, GELU) for the audio encoder and
// the token-path GEMMs.  Two instantiations keep each one small enough for the instruction cache.
#define UC_MMA(...) do { if constexpr (CTA2) mma2_bf16_ss_pred(__VA_ARGS__); else mma_bf16_ss_pred(__VA_ARGS__); } while (0)
#define UC_COMMIT(...) do { if constexpr (CTA2) mma2_commit_pred(__VA_ARGS__); else mma_commit_pred(__VA_ARGS__); } while (0)
template <int MODE>
__global__ void __launch_bounds__(UC_THREADS, 1) umma_conv_kernel(const __grid_constant__ UmmaConvP p) {
  // MODE 3 (p.cta2): the lean epilogue on CTA pairs (cluster of 2, tcgen05 cta_group::2).  The two CTAs of a pair take the tiles
  // 2j and 2j+1 (own A rows, own accumulator, own epilogue) but each stages only HALF of the weight columns; the leader's MMA
  // (M = 256) reads both halves.  A 64-column MMA then reads 4 KB of A + 1 KB of B from each SM's shared memory instead of 4 + 2:
  // 40 instead of 48 cycles of the 128 B/cycle read port that bounds the Cout = 64 layers (stem, layer1).
  constexpr bool GENERIC = MODE == 1, CTA2 = MODE == 3;
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t full_bar[8], empty_bar[8], tfull_bar[2], tempty_bar[2];
  __shared__ uint64_t full2_bar[8], tempty2_bar[2];      // CTA2, leader's copies used: peer's stage landed / peer's epilogue drained
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float bias_s[256];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool dbg = p.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0;
  if (dbg && tid == 0) p.dbg[0] = clock64();
  const int S = p.MT * 128;
  const uint32_t stage_bytes = p.a_stage_bytes + p.w_stage_bytes;
  const int num_tiles = (int)((p.g.P_total + S - 1) / S);
  const uint32_t cta_rank = CTA2 ? cluster_ctarank() : 0u;
  const int slice = blockIdx.y;
  const bool fold = p.fold != 0;                                    // (folded conv: grid.y = (output position, Cout slice))
  const int nst = fold ? (int)p.fslice[slice].nst : p.nst_tile;    // ring stages per tile of this CTA's column slice
  const int ch0 = (fold ? (int)p.fslice[slice].col : slice) * p.Cout;
  const int bcols = CTA2 ? p.Cout >> 1 : p.Cout;         // weight columns in this CTA's shared memory
  const uint32_t buf_cols = (uint32_t)(p.MT * p.Cout);
  // tile walk: tile_first, tile_first + tile_step, ... < tile_end; tile i covers positions i*S .. + S
  int tile_first = blockIdx.x, tile_step = gridDim.x, tile_end = num_tiles;
  if constexpr (CTA2) {   // the walk runs over tile PAIRS; this CTA's tile of pair j is 2j + rank (the last pair may repeat the last tile)
    tile_first = blockIdx.x >> 1; tile_step = gridDim.x >> 1; tile_end = (num_tiles + 1) >> 1;
  }
  auto tile_p0 = [&](int tile) -> int64_t {
    if constexpr (CTA2) return (int64_t)min(2 * tile + (int)cta_rank, num_tiles - 1) * S;
    return (int64_t)tile * S;
  };

  const int n_issuers = p.issuers;          // MMA-issuing warps (M-tiles are independent accumulators), chosen on the host
  if (tid == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], n_issuers); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], n_issuers); mbar_init(&tempty_bar[i], UC_EPI_WARPS); mbar_init(&tempty2_bar[i], UC_EPI_WARPS); }
    for (int i = 0; i < p.stages; ++i) mbar_init(&full2_bar[i], 1);
    fence_barrier_init();
  }
  if (warp == UC_EPI_WARP0) {
    if constexpr (CTA2) { tmem_alloc2(&tmem_base_s, p.tmem_cols); tmem_relinquish2(); }
    else { tmem_alloc(&tmem_base_s, p.tmem_cols); tmem_relinquish(); }
  }
  for (int i = tid; i < p.Cout; i += UC_THREADS) bias_s[i] = p.bias ? p.bias[ch0 + i] : 0.0f;
  // Lean instantiations: the bias enters the accumulator through ONE extra MMA per M-tile instead of 8 shared-memory loads + 32
  // additions per epilogue step (the epilogue warps, not the tensor pipe, bounded the stem and the residual convolutions once the
  // CTA pairs had shortened the MMAs).  A = 128 rows x (1, 1, 1, 0, ...) (both K halves alias the same 2 KB: LBO = 0),
  // B = per column (hi, mid, lo, 0, ...) with b = hi + mid + lo in bf16 parts (24 mantissa bits: exact), second K half zero.
  uint8_t* const bias_a = smem + (size_t)p.stages * stage_bytes + (((size_t)p.nst_tile * sizeof(UcStageDesc) + 127) & ~(size_t)127);
  uint8_t* const bias_b = bias_a + 2048;
  if constexpr (!GENERIC) {
    for (int i = tid; i < 128; i += UC_THREADS) reinterpret_cast<uint4*>(bias_a)[i] = make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u);
    for (int i = tid; i < 2 * bcols; i += UC_THREADS) {
      uint4 o = make_uint4(0u, 0u, 0u, 0u);
      if (i < bcols && p.bias) {
        const float b = p.bias[ch0 + (int)cta_rank * bcols + i];
        const __nv_bfloat16 hi = __float2bfloat16_rn(b);
        const float r1 = b - __bfloat162float(hi);
        const __nv_bfloat16 mid = __float2bfloat16_rn(r1);
        const __nv_bfloat16 lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
        o.x = (uint32_t)__bfloat16_as_ushort(hi) | ((uint32_t)__bfloat16_as_ushort(mid) << 16);
        o.y = (uint32_t)__bfloat16_as_ushort(lo);
      }
      reinterpret_cast<uint4*>(bias_b)[i] = o;
    }
    fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core's operand reads
  }
  // stage program -> shared memory (one 16-byte piece per thread)
  UcStageDesc* prog = reinterpret_cast<UcStageDesc*>(smem + (size_t)p.stages * stage_bytes);
  {
    const uint4* psrc = reinterpret_cast<const uint4*>(p.prog + (fold ? (int)p.fslice[slice].prog_off : 0));
    uint4* pdst = reinterpret_cast<uint4*>(prog);
    for (int i = tid; i < nst * 4; i += UC_THREADS) pdst[i] = psrc[i];
  }
  tc_fence_before();
  if constexpr (CTA2) cluster_sync_all();   // (the peer's barriers are initialised before anything arrives on them remotely)
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  if (dbg && tid == 0) p.dbg[1] = clock64();   // prologue done

  if (warp < UC_PROD_WARPS) {
    // ------------------------------------------------ producers (every warp runs the loop; lane 0 of each issues its share)
    // Stage k of the CTA's stream (k counts across tiles) belongs to producer warp k % npw: the per-stage work (descriptor reads,
    // address arithmetic, barrier wait, ~330-cycle bulk-copy issue) then overlaps across the four warps.  Lane l issues the
    // stage's copy l, all issuing lanes in ONE converged cp.async.bulk.
    // (Parity waits cannot alias as long as a warp is never two uses of a slot ahead of the consumer: a warp reaches stage k
    // only after stage k - npw - stages completed, which covers stage k - 2*stages iff stages >= npw.)
    const int npw = min(UC_PROD_WARPS, p.stages);
    if (warp >= npw) goto done;
    const uint32_t smem_base = smem_u32(smem);
    const uint64_t slice64 = CTA2 ? (uint64_t)cta_rank : (uint64_t)slice;   // (CTA2: the packed weights hold the two column halves as slices)
    int k = 0;                                              // global stage counter at the start of the tile
    for (int tile = tile_first; tile < tile_end; tile += tile_step, k += nst) {
      const uint64_t p0_bytes = (uint64_t)tile_p0(tile) * 16u;
      // first stage of this tile owned by this warp: si = (warp - k) mod 4
      for (int si = ((warp - k) % npw + npw) % npw; si < nst; si += npw) {
        const int kk = k + si;
        const int stage = kk % p.stages;
        const uint32_t ph = (uint32_t)(kk / p.stages) & 1u;
        const UcStageDesc& d = prog[si];
        const uint32_t counts = d.counts;
        const uint32_t n_a = counts & 0xffu, n_all = n_a + ((counts >> 8) & 0xffu);
        const bool is_a = (uint32_t)lane < n_a;
        const bool mine = (uint32_t)lane < n_all;
        const uint32_t j = is_a ? ((uint32_t)lane >> 1) : ((uint32_t)lane - n_a);   // K chunk (planar A: plane lane & 1)
        const uint32_t sa = smem_base + (uint32_t)stage * stage_bytes;
        const uint64_t gsrc = is_a ? d.a_src + p0_bytes + (uint64_t)j * d.chunk_stride_b + (uint64_t)(lane & 1) * d.plane_stride_b
                                   : d.w_src + slice64 * d.w_slice_stride_b + (uint64_t)j * (uint64_t)d.w_src_step;
        const uint32_t dst = is_a ? sa + (uint32_t)lane * d.bytesA : sa + p.a_stage_bytes + j * d.w_dst_step;
        const uint32_t nbytes = is_a ? d.bytesA : d.w_copy_bytes;
        const uint32_t tx_bytes = d.tx_bytes;
        mbar_wait(&empty_bar[stage], ph ^ 1u);
        if (dbg && lane == 0 && tile == (int)blockIdx.x && si < 24) p.dbg[32 + si] = clock64();
        if (lane == 0) mbar_arrive_expect_tx(&full_bar[stage], tx_bytes);
        __syncwarp();                                        // the expectation is registered before any completion can arrive
        if (mine) bulk_s2(dst, reinterpret_cast<const void*>(gsrc), nbytes, &full_bar[stage]);
        __syncwarp();
        if (dbg && lane == 0 && tile == (int)blockIdx.x && si < 8) p.dbg[56 + si] = clock64();   // copies issued
      }
    }
  } else if (warp < UC_MMA_WARP0 + UC_MMA_WARPS) {
    // ------------------------------------------------ MMA issuers (whole warp runs the loop; one elected lane issues)
    if (warp - UC_MMA_WARP0 >= n_issuers) goto done;
    if constexpr (CTA2) {
      if (cta_rank != 0) {
        // peer CTA: no MMAs are issued here.  One warp relays "this CTA's stage has landed" to the leader's full2 barrier.
        if (warp != UC_MMA_WARP0) goto done;
        int stage = 0;
        uint32_t ph = 0;
        for (int tile = tile_first; tile < tile_end; tile += tile_step)
          for (int si = 0; si < nst; ++si) {
            mbar_wait(&full_bar[stage], ph);
            if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&full2_bar[stage]), 0u));
            __syncwarp();
            if (++stage == p.stages) { stage = 0; ph ^= 1u; }
          }
        goto done;
      }
    }
    // (the warp index as a value ptxas knows to be warp-uniform: everything derived from it — TMEM column, M-tile offset of the A
    // descriptor — then lives in uniform registers; derived from threadIdx.x it cost an R2UR.BROADCAST per operand per MMA)
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const int mt_n = p.MT / n_issuers;                                               // this warp's M-tiles: [mt_lo, mt_lo + mt_n)
    const int mt_lo = (warp_u - UC_MMA_WARP0) * mt_n;
    // One thread feeds the tensor core: keep the per-instruction work to a few 32-bit adds.  A descriptor is
    // (constant high part) | (start address >> 4); tap / M-tile / K-chunk offsets are added in 16-byte units.
    const uint32_t idesc = idesc_bf16(CTA2 ? 256 : 128, p.Cout);
    const uint32_t smem_base = smem_u32(smem);
    const uint64_t desc_hi64 = ((uint64_t)8 << 32) | ((uint64_t)1 << 46);          // high word: SBO = 128 B, descriptor version 1
    const uint32_t b_lbo = (uint32_t)bcols << 16;                                  // LBO(B) = (staged) Cout * 16 B
    const uint32_t tap_w = (uint32_t)bcols * 2u;                                   // Cout * 32 B per tap, in 16 B units
    const uint32_t leader = elect_one() ? 1u : 0u;                                 // the lane that issues (fixed for the whole kernel)
    int stage = 0, lt = 0, dbg_it = 0;
    uint32_t ph = 0;
    for (int tile = tile_first; tile < tile_end; ++lt, tile += tile_step) {
      const int buf = p.nbuf == 2 ? (lt & 1) : 0;
      const uint32_t use = p.nbuf == 2 ? ((uint32_t)lt >> 1) : (uint32_t)lt;   // how many times this buffer was used before
      const uint32_t tb = tmem_base + (uint32_t)buf * buf_cols + (uint32_t)(mt_lo * p.Cout);
      mbar_wait(&tempty_bar[buf], (use & 1u) ^ 1u);   // epilogue has drained this accumulator buffer
      if constexpr (CTA2) mbar_wait_cluster(&tempty2_bar[buf], (use & 1u) ^ 1u);   // ... and so has the peer's
      tc_fence_after();
      uint32_t acc = 0;
      if constexpr (!GENERIC) {
        // accumulators start as the bias (overwrite: accumulate = 0)
        const uint64_t da = desc_hi64 | (uint64_t)(smem_u32(bias_a) >> 4);                   // LBO = 0
        const uint64_t db = desc_hi64 | (uint64_t)((smem_u32(bias_b) >> 4) | b_lbo);
        UC_MMA(tb, da, db, idesc, 0u, leader);
        if (mt_n > 1) UC_MMA(tb + (uint32_t)p.Cout, da, db, idesc, 0u, leader);
        if (mt_n > 2) {
          UC_MMA(tb + 2u * (uint32_t)p.Cout, da, db, idesc, 0u, leader);
          UC_MMA(tb + 3u * (uint32_t)p.Cout, da, db, idesc, 0u, leader);
        }
        acc = 1u;
      }
      // One iteration per ring stage of the tile's stage program (the program fixes the band and the K chunks of every stage, so
      // a folded conv's slices run their own band lists).  The loop reads the parameter block with warp-uniform indices (the
      // stage's counts word is broadcast from lane 0, which ptxas treats as uniform) and runs on every lane; only the MMA /
      // commit instructions are predicated on the elected lane, so the descriptor arithmetic stays in uniform registers instead
      // of being moved there (R2UR) for every instruction.
      for (int si = 0; si < nst; ++si) {
        const uint32_t counts = __shfl_sync(0xffffffffu, prog[si].counts, 0);
        const int b = (int)((counts >> 16) & 0xffu), nc = (int)(counts >> 24);
        const UcBand& bd = p.bands[b];
        const int ntaps = bd.ntaps;
        const uint32_t unitsA = (uint32_t)(S + bd.len_extra);
        const uint32_t a_lbo = (bd.toeplitz ? 1u : unitsA) << 16;     // low descriptor word = LBO << 16 | start address >> 4
        const uint32_t a_chunk = bd.toeplitz ? 2u : 2u * unitsA;
        const uint32_t w_chunk = (uint32_t)ntaps * tap_w;
        mbar_wait(&full_bar[stage], ph);
        if constexpr (CTA2) mbar_wait_cluster(&full2_bar[stage], ph);   // the peer's A rows and weight half have landed too
        tc_fence_after();
        if (dbg && warp == UC_MMA_WARP0 && lane == 0 && acc == 0 && lt == 0) p.dbg[2] = clock64();   // first stage landed
        if (dbg && warp == UC_MMA_WARP0 && lane == 0 && lt == 0 && dbg_it < 24) p.dbg[8 + dbg_it++] = clock64();
        const uint32_t sa = ((smem_base + (uint32_t)stage * stage_bytes) >> 4) + (uint32_t)mt_lo * 128u;
        const uint32_t sw = ((smem_base + (uint32_t)stage * stage_bytes + p.a_stage_bytes) >> 4) | b_lbo;
        if (ntaps == 1) {
          // Linear layers (one tap per band): one MMA per K chunk, descriptors advance by constant steps
          uint32_t at = (sa | a_lbo) + (uint32_t)bd.rel[0], wj = sw;
#pragma unroll 1
          for (int j = 0; j < nc; ++j, at += a_chunk, wj += w_chunk) {
            const uint64_t da = desc_hi64 | (uint64_t)at, db = desc_hi64 | (uint64_t)wj;
            UC_MMA(tb, da, db, idesc, acc, leader);
            if (mt_n > 1) UC_MMA(tb + (uint32_t)p.Cout, da + 128u, db, idesc, acc, leader);
            acc = 1u;
          }
        } else
        for (int j = 0; j < nc; ++j) {
          const uint32_t aj = (sa + (uint32_t)j * a_chunk) | a_lbo;
          uint32_t wj = sw + (uint32_t)j * w_chunk;
#pragma unroll 1
          for (int tp = 0; tp < ntaps; ++tp) {   // (not unrolled: the kernel must stay inside the instruction cache)
            const uint32_t at = aj + (uint32_t)bd.rel[tp];
            const uint64_t da = desc_hi64 | (uint64_t)at, db = desc_hi64 | (uint64_t)wj;
            UC_MMA(tb, da, db, idesc, acc, leader);
            if (mt_n > 1) UC_MMA(tb + (uint32_t)p.Cout, da + 128u, db, idesc, acc, leader);
            if (mt_n > 2) {
              UC_MMA(tb + 2u * (uint32_t)p.Cout, da + 256u, db, idesc, acc, leader);
              UC_MMA(tb + 3u * (uint32_t)p.Cout, da + 384u, db, idesc, acc, leader);
            }
            acc = 1u;
            wj += tap_w;
          }
        }
        UC_COMMIT(&empty_bar[stage], leader);  // frees the stage once the MMAs that read it have completed
        if (++stage == p.stages) { stage = 0; ph ^= 1u; }
      }
      UC_COMMIT(&tfull_bar[buf], leader);   // accumulator of this tile complete -> epilogue
      if (dbg && warp == UC_MMA_WARP0 && lane == 0 && lt == 0) p.dbg[3] = clock64();   // all MMAs of the first tile issued
    }
  } else {
    // ------------------------------------------------ epilogue warps (TMEM lane quarter = warp % 4; thread == tile row)
    const int quarter = warp & 3;
    const int half = (warp - UC_EPI_WARP0) >> 2;                 // which 32-column chunks this warp handles (even / odd)
    const float act_lo = p.act == ACT_RELU ? 0.0f : -INFINITY;   // ReLU as one FMNMX; GELU (token GEMMs only) branches once per chunk
    const int rowt = quarter * 32 + lane;
    int lt = 0;
    for (int tile = tile_first; tile < tile_end; ++lt, tile += tile_step) {
      const int buf = p.nbuf == 2 ? (lt & 1) : 0;
      const uint32_t use = p.nbuf == 2 ? ((uint32_t)lt >> 1) : (uint32_t)lt;
      const uint32_t tb = tmem_base + (uint32_t)buf * buf_cols + ((uint32_t)(quarter * 32) << 16);
      const int64_t P0 = tile_p0(tile);
      mbar_wait(&tfull_bar[buf], use & 1u);
      tc_fence_after();
      if (dbg && warp == UC_EPI_WARP0 && lane == 0 && lt == 0) p.dbg[4] = clock64();   // first accumulator complete
      // Lean path with several M-tiles per tile: the two warps of a TMEM lane quarter take alternate M-tiles and all columns
      // (one position decode per M-tile and thread instead of two); otherwise they split the columns.
      const bool split_m = !GENERIC && p.MT >= 2;
      // (the lean epilogue works in 32-column steps: with a single M-tile the columns are split only if both halves are whole
      // steps, otherwise the first warp of the quarter takes all of them)
      const bool split_c = !split_m && (GENERIC || (p.Cout & 63) == 0);
      const int m_end = (!split_m && !split_c && half == 1) ? 0 : p.MT;
      for (int m = split_m ? half : 0; m < m_end; m += split_m ? 2 : 1) {
        const int64_t P = P0 + (int64_t)m * 128 + rowt;
        int n = 0, t = 0, h = 0, w = 0;
        const bool valid = (p.skip & 8) ? true : uc_decode(p.g, P, n, t, h, w);   // (skip bit 3: timing experiment)
        if (fold) { h = p.fslice[slice].h; w = p.fslice[slice].w; }               // (row geometry: P is the frame row)
        const bool inrange = P < p.g.P_total;
        const int64_t outer = valid ? ((int64_t)n * p.g.T + t) * p.g.H + h : 0;
        int64_t dst = P * 8;
        if (valid && p.y_mode == UC_Y_PARITY)
          dst = (int64_t)((h & 1) * 2 + (w & 1)) * p.y_set_stride + uc_flat(p.g2, n, t, h >> 1, w >> 1) * 8;
        else if (valid && p.y_mode == UC_Y_PARITY_H)
          dst = (int64_t)((h & 1) * 2) * p.y_set_stride + uc_flat(p.g2, n, t, h >> 1, w) * 8;
        else if (valid && p.y_mode == UC_Y_FOLD)
          dst = (int64_t)(h * p.ymap_W + w) * p.y_set_stride + uc_flat(p.g2, n, t, 0, 0) * 8;
        else if (valid && p.y_mode == UC_Y_MAP)
          dst = uc_flat(p.g2, n, t, h, w) * 8;
        const bool store_planar = ((p.y_mode == UC_Y_PLAIN && inrange) || (p.y_mode >= UC_Y_PARITY && valid)) && !(p.skip & 4);   // (skip bit 2: timing experiment)
        // this warp's columns: [half*Cout/2, (half+1)*Cout/2), or all of them when the warps split the M-tiles
        const int cbeg = split_c ? half * (p.Cout >> 1) : 0, cend = split_c ? cbeg + (p.Cout >> 1) : p.Cout;
        if constexpr (!GENERIC) {
          // lean path (Cout % 32 == 0, checked on the host): 32 columns per step.  One 32-column TMEM load, the bias (shared
          // memory) and the residual (global) are fetched before the single wait, the activation rides on the bf16 conversion
          // (cvt.rn.relu), pads are zeroed by a mask on the packed words.  ~110 instructions per step instead of ~450: the stem and
          // the hf front convolution were bound by the instruction issue of these eight warps, not by the tensor pipe.
          char* yp = reinterpret_cast<char*>(p.y + (int64_t)((ch0 + cbeg) >> 3) * p.y_plane_stride + dst);
          const char* rp = reinterpret_cast<const char*>(p.res + (int64_t)((ch0 + cbeg) >> 3) * p.res_plane_stride + P * 8);
          const int64_t yps = p.y_plane_stride * 2, rps = p.res_plane_stride * 2;
          const bool has_res = p.res != nullptr;   // (warp-uniform)
          const bool relu = p.act == ACT_RELU;
          const uint32_t vmask = valid ? 0xffffffffu : 0u;
          uint32_t ta = tb + (uint32_t)(m * p.Cout + cbeg);
#pragma unroll 1
          for (int c = cbeg; c < cend; c += 32, yp += 4 * yps, rp += 4 * rps, ta += 32) {
            float v[32];
            uint4 rr[4];
            tmem_ld32(ta, v);        // (the bias is already in the accumulator: see the MMA issuer)
            if (has_res) {
#pragma unroll
              for (int q = 0; q < 4; ++q) rr[q] = valid ? *reinterpret_cast<const uint4*>(rp + q * rps) : make_uint4(0, 0, 0, 0);
            }
            tmem_ld_wait();
            if (has_res) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                float f[8];
                unpack8(rr[q], f);
#pragma unroll
                for (int e = 0; e < 8; ++e) v[8 * q + e] += f[e];
              }
            }
            if (store_planar) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                uint4 o = relu ? pack8_relu(v + 8 * q) : pack8(v + 8 * q);
                o.x &= vmask; o.y &= vmask; o.z &= vmask; o.w &= vmask;
                *reinterpret_cast<uint4*>(yp + q * yps) = o;
              }
            }
          }
        } else {
        // generic path (Cout % 64 == 0, at most one kind of residual — checked on the host): 32 columns per step.  One 32-column
        // TMEM load; the step's residuals (bf16 hi [+ lo] planes, or fp32 rows) are fetched before the single wait, so the
        // global-load latency and the TMEM round trip are paid once per step instead of once per 8 columns.
        const float* r32row = p.res32 ? p.res32 + (outer * p.g.W + w) * p.res32_ld + ch0 : nullptr;
        float* y32row = p.y32 ? p.y32 + (outer * p.y32_outer_stride + w + p.y32_row_off) * p.y32_ld + ch0 : nullptr;
        const bool use_res = valid && p.res != nullptr, use_lo = use_res && p.res_lo != nullptr, use_r32 = valid && p.res32 != nullptr;
#pragma unroll 1
        for (int c0 = cbeg; c0 < cend; c0 += 32) {
          float v[32];
          uint4 pre[8];
          tmem_ld32(tb + (uint32_t)(m * p.Cout + c0), v);
          if (use_res) {
            const int64_t roff = (int64_t)((ch0 + c0) >> 3) * p.res_plane_stride + P * 8;
#pragma unroll
            for (int q = 0; q < 4; ++q) pre[q] = *reinterpret_cast<const uint4*>(p.res + roff + (int64_t)q * p.res_plane_stride);
            if (use_lo) {
#pragma unroll
              for (int q = 0; q < 4; ++q) pre[4 + q] = *reinterpret_cast<const uint4*>(p.res_lo + roff + (int64_t)q * p.res_plane_stride);
            }
          } else if (use_r32) {
#pragma unroll
            for (int q = 0; q < 8; ++q) pre[q] = *reinterpret_cast<const uint4*>(r32row + c0 + 4 * q);
          }
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int c = c0 + 8 * q;
            F8 x;
#pragma unroll
            for (int e = 0; e < 8; ++e) x.v[e] = v[8 * q + e];
            if (valid) {
              const float4 b0 = *reinterpret_cast<const float4*>(&bias_s[c]);
              const float4 b1 = *reinterpret_cast<const float4*>(&bias_s[c + 4]);
              x.v[0] += b0.x; x.v[1] += b0.y; x.v[2] += b0.z; x.v[3] += b0.w; x.v[4] += b1.x; x.v[5] += b1.y; x.v[6] += b1.z; x.v[7] += b1.w;
              if (use_res) {
                float f[8];
                unpack8(pre[q], f);
#pragma unroll
                for (int e = 0; e < 8; ++e) x.v[e] += f[e];
                if (use_lo) {
                  unpack8(pre[4 + q], f);
#pragma unroll
                  for (int e = 0; e < 8; ++e) x.v[e] += f[e];
                }
              } else if (use_r32) {
                const uint4 q0 = pre[2 * q], q1 = pre[2 * q + 1];
                x.v[0] += __uint_as_float(q0.x); x.v[1] += __uint_as_float(q0.y); x.v[2] += __uint_as_float(q0.z); x.v[3] += __uint_as_float(q0.w);
                x.v[4] += __uint_as_float(q1.x); x.v[5] += __uint_as_float(q1.y); x.v[6] += __uint_as_float(q1.z); x.v[7] += __uint_as_float(q1.w);
              }
              if (p.act == ACT_GELU) {
                x = gelu8(x);   // (out of line: 32 inlined erff per step would not fit the instruction cache)
              } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) x.v[e] = fmaxf(x.v[e], act_lo);
              }
              if (y32row) {
                float4* o = reinterpret_cast<float4*>(y32row + c);
                o[0] = make_float4(x.v[0], x.v[1], x.v[2], x.v[3]);
                o[1] = make_float4(x.v[4], x.v[5], x.v[6], x.v[7]);
              }
            } else {
#pragma unroll
              for (int e = 0; e < 8; ++e) x.v[e] = 0.0f;
            }
            if (store_planar) {
              const uint4 hi4 = pack8(x.v);
              const int64_t off = (int64_t)((ch0 + c) >> 3) * p.y_plane_stride + dst;
              *reinterpret_cast<uint4*>(p.y + off) = hi4;
              if (p.ylo) {
                float hf[8];
                unpack8(hi4, hf);
#pragma unroll
                for (int e = 0; e < 8; ++e) hf[e] = x.v[e] - hf[e];
                *reinterpret_cast<uint4*>(p.ylo + off) = pack8(hf);
              }
            }
          }
        }
        }
      }
      // all TMEM reads of this warp are complete (wait::ld above): hand the buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CTA2 && cta_rank != 0) mbar_arrive_cluster(mapa_shared(smem_u32(&tempty2_bar[buf]), 0u));
        else mbar_arrive(&tempty_bar[buf]);
      }
      if (dbg && warp == UC_EPI_WARP0 && lane == 0 && lt == 0) p.dbg[5] = clock64();   // first epilogue done
    }
  }
done:
  tc_fence_before();
  if constexpr (CTA2) cluster_sync_all();   // (both CTAs are done with the pair's tensor memory and barriers)
  else __syncthreads();
  if (warp == UC_EPI_WARP0) {
    if constexpr (CTA2) tmem_dealloc2(tmem_base, p.tmem_cols);
    else tmem_dealloc(tmem_base, p.tmem_cols);
  }
  if (dbg && tid == 0) { p.dbg[6] = clock64(); p.dbg[7] = num_tiles; }
}

UcStageDesc umma_conv_stage(const UmmaConvP& p, const UcGroup& g, const UcBand& bd, int band, int c0, int col) {
  const int S = p.MT * 128;
  const int bcols = p.cta2 ? p.Cout / 2 : p.Cout;   // weight columns one CTA stages
  const int nc = std::min(p.kpack, g.k16 - c0);
  UcStageDesc d;
  const uint32_t bytesW = (uint32_t)bd.ntaps * (uint32_t)bcols * 32u;
  d.bytesA = bd.toeplitz ? (uint32_t)(S + bd.len_extra + 1 + 2 * (nc - 1)) * 16u : (uint32_t)(S + bd.len_extra) * 16u;
  uint32_t n_a = bd.toeplitz ? 1u : 2u * (uint32_t)nc;   // Toeplitz: the K chunks are 32-byte shifts of one row region
  // a band that holds all taps of its group (Linear layers, the fused 1x1 downsample): the weights of consecutive K chunks are
  // contiguous -> one copy
  const bool w_merged = bd.ntaps == g.taps_total;
  uint32_t n_w = w_merged ? 1u : (uint32_t)nc;
  d.w_copy_bytes = w_merged ? (uint32_t)nc * bytesW : bytesW;
  d.w_dst_step = bytesW;
  // (p.skip: timing experiments only — bit 0 drops the A copies, bit 1 the W copies; results are then garbage)
  if (p.skip & 1) n_a = 0;
  if (p.skip & 2) n_w = 0;
  d.tx_bytes = n_a * d.bytesA + (n_w ? (uint32_t)nc * bytesW : 0u);
  d.a_src = reinterpret_cast<uint64_t>(bd.base + (int64_t)c0 * bd.chunk_stride + (int64_t)bd.start * 8);
  d.chunk_stride_b = (uint64_t)bd.chunk_stride * 2u;
  d.plane_stride_b = (uint64_t)bd.plane_stride * 2u;
  // weight piece j of the stage is the packed block [chunk c0 + j][taps of this band]: pieces are taps_total * Cout * 32 B apart
  d.w_src = reinterpret_cast<uint64_t>(p.w + g.w_off + (col > 0 ? (int64_t)col * g.slice_stride : 0) +
                                       ((int64_t)c0 * g.taps_total + bd.tap_begin) * (int64_t)bcols * 16);
  d.w_slice_stride_b = col >= 0 ? 0u : (uint64_t)g.slice_stride * 2u;
  d.w_src_step = (uint32_t)g.taps_total * (uint32_t)bcols * 32u;
  d.counts = n_a | (n_w << 8) | ((uint32_t)band << 16) | ((uint32_t)nc << 24);
  return d;
}

void umma_conv_build_program(const UmmaConvP& p, UcStageDesc* out) {
  int s = 0;
  for (int gi = 0; gi < p.ngroups; ++gi) {
    const UcGroup& g = p.groups[gi];
    for (int c0 = 0; c0 < g.k16; c0 += p.kpack)
      for (int b = g.band_begin; b < g.band_end; ++b) out[s++] = umma_conv_stage(p, g, p.bands[b], b, c0);
  }
}

size_t umma_conv_smem_bytes(const UmmaConvP& p) {
  size_t b = (size_t)p.stages * (p.a_stage_bytes + p.w_stage_bytes) + (size_t)p.nst_tile * sizeof(UcStageDesc) + 1024;
  return b + umma_conv_extra_smem_bytes(p);
}
int umma_conv_stage_desc_bytes() { return (int)sizeof(UcStageDesc); }
static bool uc_is_generic(const UmmaConvP& p);
// shared memory behind the stage program: the bias operand tiles of the lean instantiations
size_t umma_conv_extra_smem_bytes(const UmmaConvP& p) {
  if (uc_is_generic(p)) return 0;
  return 128 + 2048 + (size_t)(p.cta2 ? p.Cout / 2 : p.Cout) * 32u;
}

static bool uc_is_generic(const UmmaConvP& p) {
  return p.y32 || p.res32 || p.ylo || p.res_lo || p.act == ACT_GELU || p.y_mode == UC_Y_NONE || (p.Cout & 31);   // (the lean epilogue works in 32-column steps)
}
const char* umma_conv_config_error(const UmmaConvP& p) {
  if (2 * p.kpack + p.kpack > 32) return "K chunks per stage exceed the producer lanes";
  if (p.res && p.res32) return "bf16 and fp32 residuals are mutually exclusive";
  if (uc_is_generic(p) && (p.Cout & 63)) return "the generic epilogue needs a column slice that is a multiple of 64";
  if (p.MT / p.issuers > 4 || p.MT % p.issuers) return "unsupported M-tiles per issuing warp";
  if (p.fold && (uc_is_generic(p) || p.cta2 || p.res || p.MT > 4))
    return "folded convolutions need the lean epilogue, no residual, single CTAs and at most 4 M-tiles";
  if (p.cta2 && (uc_is_generic(p) || (p.Cout & 31))) return "CTA pairs need the lean epilogue and a multiple of 32 columns";
  return nullptr;
}

// Function attributes are per device: lsd_create calls this once with the handle's device current.
cudaError_t umma_conv_device_init() {
  // the opt-in limit (227 KB) covers static + dynamic shared memory; ~3.7 KB is static (barriers, bias, band / group tables)
  cudaError_t e = cudaFuncSetAttribute(umma_conv_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 223 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(umma_conv_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 223 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(umma_conv_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 223 * 1024);
  if (e == cudaSuccess) e = video_rows_device_init();
  return e;
}

void launch_umma_conv(const UmmaConvP& p, int n_slices, cudaStream_t s, int num_sms, int max_ctas) {
  if (const char* why = umma_conv_config_error(p)) { fprintf(stderr, "umma_conv: %s\n", why); abort(); }   // (callers check first)
  const int S = p.MT * 128;
  const int tiles = (int)((p.g.P_total + S - 1) / S);
  // persistent grid: one CTA per SM (per Cout slice), each walking tiles with stride gridDim.x
  const int budget = (max_ctas > 0 && max_ctas < num_sms) ? max_ctas : num_sms;   // side-stream launches leave SMs to the main stream
  int gx = (budget + n_slices - 1) / n_slices;
  gx = gx < 1 ? 1 : (gx > tiles ? tiles : gx);
  const bool generic = uc_is_generic(p);
  if (p.cta2) {
    // CTA pairs: an even grid of clusters of 2 (one pair per TPC), each pair walking tile pairs
    if (n_slices != 1) { fprintf(stderr, "umma_conv: CTA pairs take one column slice\n"); abort(); }
    const int pairs = (tiles + 1) / 2;
    int gp = budget / 2;
    gp = gp < 1 ? 1 : (gp > pairs ? pairs : gp);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * gp, 1, 1);
    cfg.blockDim = dim3(UC_THREADS, 1, 1);
    cfg.dynamicSmemBytes = umma_conv_smem_bytes(p);
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, umma_conv_kernel<3>, p);
    count_launch();
    return;
  }
  if (p.fold) gx = tiles;   // folded convs: one tile per CTA; the heaviest slices come first and the block scheduler balances the rest
  if (generic) umma_conv_kernel<1><<<dim3(gx, n_slices), UC_THREADS, umma_conv_smem_bytes(p), s>>>(p);
  else umma_conv_kernel<0><<<dim3(gx, n_slices), UC_THREADS, umma_conv_smem_bytes(p), s>>>(p);
  count_launch();
}

// ================================================================================================
// planar-layout glue kernels (memory-bound, 16-byte accesses, one thread per (position, 8-channel chunk))
// ================================================================================================
__global__ void pack_planar_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int64_t plane_stride, int64_t set_stride,
                                   UcGeom g, UcGeom g2, int C, int parity, int64_t total) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  // position-major within a chunk so that a warp writes 512 contiguous bytes of one plane
  const int64_t npos = (int64_t)g.N * g.T * g.H * g.W;
  const int chunk = (int)(i / npos);
  int64_t r = i - (int64_t)chunk * npos;
  const int w = (int)(r % g.W); r /= g.W;
  const int h = (int)(r % g.H); r /= g.H;
  const int t = (int)(r % g.T);
  const int n = (int)(r / g.T);
  const float* src = x + ((((int64_t)n * g.T + t) * g.H + h) * g.W + w) * C + chunk * 8;
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = src[e];
  int64_t dst;
  if (parity) dst = (int64_t)((h & 1) * 2 + (w & 1)) * set_stride + uc_flat(g2, n, t, h >> 1, w >> 1) * 8;
  else dst = uc_flat(g, n, t, h, w) * 8;
  *reinterpret_cast<uint4*>(y + (int64_t)chunk * plane_stride + dst) = pack8(v);
}
void launch_pack_planar(const float* x, __nv_bfloat16* y, int64_t plane_stride, int64_t set_stride, UcGeom g, UcGeom g2, int C,
                        int parity, cudaStream_t s) {
  const int64_t total = (int64_t)g.N * g.T * g.H * g.W * (C / 8);
  if (total == 0) return;
  pack_planar_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(x, y, plane_stride, set_stride, g, g2, C, parity, total);
  count_launch();
}

__global__ void unpack_planar_kernel(const __nv_bfloat16* __restrict__ x, int64_t plane_stride, UcGeom g, int C, float* __restrict__ y,
                                     int ld, int64_t total) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int nch = C / 8;
  const int chunk = (int)(i % nch);
  int64_t r = i / nch;
  const int64_t row = r;
  const int w = (int)(r % g.W); r /= g.W;
  const int h = (int)(r % g.H); r /= g.H;
  const int t = (int)(r % g.T);
  const int n = (int)(r / g.T);
  const uint4 v = *reinterpret_cast<const uint4*>(x + (int64_t)chunk * plane_stride + uc_flat(g, n, t, h, w) * 8);
  float f[8];
  unpack8(v, f);
  float4* o = reinterpret_cast<float4*>(y + row * ld + chunk * 8);
  o[0] = make_float4(f[0], f[1], f[2], f[3]);
  o[1] = make_float4(f[4], f[5], f[6], f[7]);
}
void launch_unpack_planar(const __nv_bfloat16* x, int64_t plane_stride, UcGeom g, int C, float* y, int ld, cudaStream_t s) {
  const int64_t total = (int64_t)g.N * g.T * g.H * g.W * (C / 8);
  if (total == 0) return;
  unpack_planar_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(x, plane_stride, g, C, y, ld, total);
  count_launch();
}

// Introspection: any planar buffer (plain, parity-split with 4 plane sets, or folded: Hf*Wf sets in the row geometry) -> fp32
// channels-last (N, T, Hf, Wf, C)
__global__ void unpack_planar_any_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ xlo, int64_t plane_stride,
                                         int64_t set_stride, UcGeom g, int C, int sets, int Hf, int Wf, float* __restrict__ y, int64_t total) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int nch = C / 8;
  const int chunk = (int)(i % nch);
  int64_t r = i / nch;
  const int64_t row = r;
  const int w = (int)(r % Wf); r /= Wf;
  const int h = (int)(r % Hf); r /= Hf;
  const int t = (int)(r % g.T);
  const int n = (int)(r / g.T);
  int64_t src;
  if (sets == 1) src = uc_flat(g, n, t, h, w) * 8;
  else if (g.SL == 1 && sets == Hf * Wf) src = (int64_t)(h * Wf + w) * set_stride + uc_flat(g, n, t, 0, 0) * 8;   // folded (one set per position)
  else if (Wf == g.W) src = (int64_t)((h & 1) * 2) * set_stride + uc_flat(g, n, t, h >> 1, w) * 8;          // h-parity split
  else src = (int64_t)((h & 1) * 2 + (w & 1)) * set_stride + uc_flat(g, n, t, h >> 1, w >> 1) * 8;          // (h, w)-parity split
  src += (int64_t)chunk * plane_stride;
  float f[8];
  unpack8(*reinterpret_cast<const uint4*>(x + src), f);
  if (xlo) {
    float fl[8];
    unpack8(*reinterpret_cast<const uint4*>(xlo + src), fl);
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] += fl[e];
  }
  float4* o = reinterpret_cast<float4*>(y + row * C + chunk * 8);
  o[0] = make_float4(f[0], f[1], f[2], f[3]);
  o[1] = make_float4(f[4], f[5], f[6], f[7]);
}
void launch_unpack_planar_any(const __nv_bfloat16* x, const __nv_bfloat16* xlo, int64_t plane_stride, int64_t set_stride, UcGeom g, int C, int sets,
                              int Hf, int Wf, float* y, cudaStream_t s) {
  const int64_t total = (int64_t)g.N * g.T * Hf * Wf * (C / 8);
  if (total == 0) return;
  unpack_planar_any_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(x, xlo, plane_stride, set_stride, g, C, sets, Hf, Wf, y, total);
  count_launch();
}

// Deterministic mean: one block per (row, chunk); threads stride over the row's positions, fixed-order tree in shared memory.
__global__ void planar_mean_kernel(const __nv_bfloat16* __restrict__ x, int64_t plane_stride, UcGeom g, float* __restrict__ y, int ld,
                                   int per_window) {
  __shared__ float part[256][9];
  const int row = blockIdx.x, chunk = blockIdx.y, tid = threadIdx.x;
  const int count = per_window ? g.T * g.H * g.W : g.H * g.W;
  const int n = per_window ? row : row / g.T;
  const int t0 = per_window ? 0 : row % g.T;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = tid; i < count; i += blockDim.x) {
    const int w = i % g.W;
    const int r = i / g.W;
    const int h = r % g.H;
    const int t = t0 + r / g.H;
    const uint4 v = *reinterpret_cast<const uint4*>(x + (int64_t)chunk * plane_stride + uc_flat(g, n, t, h, w) * 8);
    float f[8];
    unpack8(v, f);
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] += f[e];
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) part[tid][e] = acc[e];
  __syncthreads();
  for (int sft = blockDim.x >> 1; sft > 0; sft >>= 1) {
    if (tid < sft) {
#pragma unroll
      for (int e = 0; e < 8; ++e) part[tid][e] += part[tid + sft][e];
    }
    __syncthreads();
  }
  if (tid < 8) y[(int64_t)row * ld + chunk * 8 + tid] = part[0][tid] / (float)count;
}
void launch_planar_mean(const __nv_bfloat16* x, int64_t plane_stride, UcGeom g, int C, float* y, int ld, int per_window, cudaStream_t s) {
  const int rows = per_window ? g.N : g.N * g.T;
  if (rows == 0) return;
  const int count = per_window ? g.T * g.H * g.W : g.H * g.W;
  int threads = 32;
  while (threads < 256 && threads < count) threads <<= 1;
  planar_mean_kernel<<<dim3(rows, C / 8), threads, 0, s>>>(x, plane_stride, g, y, ld, per_window);
  count_launch();
}

__global__ void planar_delta_kernel(const __nv_bfloat16* __restrict__ x, int64_t xs, UcGeom g, __nv_bfloat16* __restrict__ d, int64_t ds,
                                    UcGeom gd, int64_t total) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int64_t npos = (int64_t)gd.N * gd.T * gd.H * gd.W;
  const int chunk = (int)(i / npos);
  int64_t r = i - (int64_t)chunk * npos;
  const int w = (int)(r % gd.W); r /= gd.W;
  const int h = (int)(r % gd.H); r /= gd.H;
  const int t = (int)(r % gd.T);
  const int n = (int)(r / gd.T);
  float a[8], b[8], o[8];
  unpack8(*reinterpret_cast<const uint4*>(x + (int64_t)chunk * xs + uc_flat(g, n, t + 1, h, w) * 8), a);
  unpack8(*reinterpret_cast<const uint4*>(x + (int64_t)chunk * xs + uc_flat(g, n, t, h, w) * 8), b);
#pragma unroll
  for (int e = 0; e < 8; ++e) o[e] = a[e] - b[e];
  *reinterpret_cast<uint4*>(d + (int64_t)chunk * ds + uc_flat(gd, n, t, h, w) * 8) = pack8(o);
}
void launch_planar_delta(const __nv_bfloat16* x, int64_t x_plane_stride, UcGeom g, __nv_bfloat16* d, int64_t d_plane_stride, UcGeom gd,
                         int C, cudaStream_t s) {
  const int64_t total = (int64_t)gd.N * gd.T * gd.H * gd.W * (C / 8);
  if (total == 0) return;
  planar_delta_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(x, x_plane_stride, g, d, d_plane_stride, gd, total);
  count_launch();
}

// MaxPool (1,3,3)/(1,2,2)/pad(0,1,1) in planar layout.  Inputs are post-ReLU (>= 0) and the pads are zero, so reading
// the zero pad is equivalent to the reference's -inf padding except at the far edge, which is bounds-checked.
__global__ void __launch_bounds__(256) planar_maxpool_kernel(const __nv_bfloat16* __restrict__ x, int64_t xs, UcGeom gi, __nv_bfloat16* __restrict__ y,
                                                             int64_t ys, UcGeom go, const __nv_bfloat16* __restrict__ xlo,
                                                             __nv_bfloat16* __restrict__ ylo) {
  // One block per (frame, 8-channel plane); a warp takes (output row, 32-column input segment) pairs.  Lane l loads input
  // column seg*32 + l of the three rows — a warp reads 512 contiguous bytes per row, every 32-byte sector fully used (the
  // per-output 16-byte gathers of the first versions made the kernel L1-bound: 12x sector amplification) — and keeps the
  // column's vertical maximum; the 16 outputs of the segment combine columns 2w-1, 2w, 2w+1 by shuffle.
  // All index arithmetic is 32-bit relative to the frame origin.
  const int frame = blockIdx.x, chunk = blockIdx.y;
  const int n = frame / go.T, t = frame - n * go.T;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const __nv_bfloat16* xc = x + (int64_t)chunk * xs + uc_flat(gi, n, t, 0, 0) * 8;      // input pixel (0,0) of this frame
  const __nv_bfloat16* xlc = xlo ? xlo + (int64_t)chunk * xs + uc_flat(gi, n, t, 0, 0) * 8 : nullptr;
  __nv_bfloat16* yc = y + (int64_t)chunk * ys + uc_flat(go, n, t, 0, 0) * 8;
  __nv_bfloat16* ylc = ylo ? ylo + (int64_t)chunk * ys + uc_flat(go, n, t, 0, 0) * 8 : nullptr;
  auto ld = [&](int pos, float* f) {
    unpack8(*reinterpret_cast<const uint4*>(xc + pos * 8), f);
    if (xlc) {
      float fl[8];
      unpack8(*reinterpret_cast<const uint4*>(xlc + pos * 8), fl);
#pragma unroll
      for (int e = 0; e < 8; ++e) f[e] += fl[e];
    }
  };
  const int nseg = (gi.W + 31) >> 5;
  const int npairs = go.H * nseg;
  for (int pair = warp; pair < npairs; pair += nwarps) {
    const int h = pair / nseg, seg = pair - h * nseg;
    const int c = seg * 32 + lane;                         // this lane's input column
    float mv[8], ml[8];                                    // vertical max of column c; of column seg*32 - 1 (lane 0 only)
#pragma unroll
    for (int e = 0; e < 8; ++e) mv[e] = ml[e] = -INFINITY;
    const bool extra_left = lane == 0 && seg > 0;
#pragma unroll
    for (int dh = 0; dh < 3; ++dh) {
      const int hi = 2 * h - 1 + dh;
      if ((unsigned)hi >= (unsigned)gi.H) continue;
      float f[8];
      if (c < gi.W) {
        ld(hi * gi.RW + c, f);
#pragma unroll
        for (int e = 0; e < 8; ++e) mv[e] = fmaxf(mv[e], f[e]);
      }
      if (extra_left) {
        ld(hi * gi.RW + c - 1, f);
#pragma unroll
        for (int e = 0; e < 8; ++e) ml[e] = fmaxf(ml[e], f[e]);
      }
    }
    const int w = seg * 16 + lane;                         // output column of lanes 0..15
    float m[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float a = __shfl_sync(0xffffffffu, mv[e], (2 * lane) & 31);
      const float b = __shfl_sync(0xffffffffu, mv[e], (2 * lane + 1) & 31);
      const float cl = __shfl_sync(0xffffffffu, mv[e], (2 * lane - 1) & 31);
      const float left = lane == 0 ? ml[e] : cl;           // (seg == 0: ml stays -inf = the reference's padding)
      m[e] = fmaxf(fmaxf(a, b), left);
    }
    if (lane < 16 && w < go.W) {
      const int dst = (h * go.RW + w) * 8;
      const uint4 hi4 = pack8(m);
      *reinterpret_cast<uint4*>(yc + dst) = hi4;
      if (ylc) {
        float hf[8], lo[8];
        unpack8(hi4, hf);
#pragma unroll
        for (int e = 0; e < 8; ++e) lo[e] = m[e] - hf[e];
        *reinterpret_cast<uint4*>(ylc + dst) = pack8(lo);
      }
    }
  }
}
// Same result for plain bf16 tensors (no hi/lo split), one thread per pooled position: nine independent predicated 16-byte loads (the
// 3x3 window; neighbours' re-reads hit L1), no shuffles, no idle lanes at the store; the maximum is taken on packed bf16 pairs
// (HMNMX2, exact in bf16).  The warp-per-row mapping above, on packed bf16 pairs, was bound by its dependent load -> shuffle chain
// (209 us for the 811 MB of the stem's max-pool at B=64: 3.9 TB/s).
__global__ void __launch_bounds__(192) planar_maxpool_direct_kernel(const __nv_bfloat16* __restrict__ x, int64_t xs, UcGeom gi,
                                                                    __nv_bfloat16* __restrict__ y, int64_t ys, UcGeom go) {
  const int frame = blockIdx.x, chunk = blockIdx.y;
  const int n = frame / go.T, t = frame - n * go.T;
  const uint4* xc = reinterpret_cast<const uint4*>(x + (int64_t)chunk * xs + uc_flat(gi, n, t, 0, 0) * 8);
  uint4* yc = reinterpret_cast<uint4*>(y + (int64_t)chunk * ys + uc_flat(go, n, t, 0, 0) * 8);
  const uint32_t NINF2 = 0xFF80FF80u;                                   // (-inf, -inf) in bf16
  const int total = go.H * go.W;
  for (int o = threadIdx.x; o < total; o += blockDim.x) {
    const int h = o / go.W, w = o - h * go.W;
    uint4 v[9];
#pragma unroll
    for (int dh = 0; dh < 3; ++dh)
#pragma unroll
      for (int dw = 0; dw < 3; ++dw) {
        const int hi = 2 * h - 1 + dh, wi = 2 * w - 1 + dw;
        v[dh * 3 + dw] = ((unsigned)hi < (unsigned)gi.H && (unsigned)wi < (unsigned)gi.W) ? xc[hi * gi.RW + wi] : make_uint4(NINF2, NINF2, NINF2, NINF2);
      }
    uint32_t* m = reinterpret_cast<uint32_t*>(&v[0]);
#pragma unroll
    for (int k = 1; k < 9; ++k) {
      const uint32_t* r = reinterpret_cast<const uint32_t*>(&v[k]);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const __nv_bfloat162 q = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&m[e]), *reinterpret_cast<const __nv_bfloat162*>(&r[e]));
        m[e] = *reinterpret_cast<const uint32_t*>(&q);
      }
    }
    yc[h * go.RW + w] = v[0];
  }
}

void launch_planar_maxpool(const __nv_bfloat16* x, int64_t x_plane_stride, UcGeom gi, __nv_bfloat16* y, int64_t y_plane_stride, UcGeom go,
                           int C, cudaStream_t s, const __nv_bfloat16* xlo, __nv_bfloat16* ylo) {
  const int frames = go.N * go.T;
  if (frames == 0 || go.H * go.W == 0) return;
  if (!xlo && !ylo) planar_maxpool_direct_kernel<<<dim3((unsigned)frames, (unsigned)(C / 8)), 192, 0, s>>>(x, x_plane_stride, gi, y, y_plane_stride, go);
  else planar_maxpool_kernel<<<dim3((unsigned)frames, (unsigned)(C / 8)), 256, 0, s>>>(x, x_plane_stride, gi, y, y_plane_stride, go, xlo, ylo);
  count_launch();
}

// One block (32 x 8 threads) per (n, t, band of VR_ROWS image rows): the band (+1 halo row/column on every side) is staged
// in shared memory with coalesced, batched loads and no integer divisions, and each thread
// produces pixel pairs (16-byte units) of both row buffers.
constexpr int VR_ROWS = 8;
// uint8 crops are scaled exactly like the reference: astype(float32) / 255.0 (video.py:552-556)
template <typename T> __device__ __forceinline__ float vr_norm(float x) { return x; }
template <> __device__ __forceinline__ float vr_norm<uint8_t>(float x) { return x / 255.0f; }
template <typename T, int LAYOUT>
__global__ void __launch_bounds__(256) video_rows_kernel(const T* __restrict__ video, const float* __restrict__ lapw,
                                                         __nv_bfloat16* __restrict__ xs, __nv_bfloat16* __restrict__ xl, int64_t set_stride,
                                                         UcGeom g, int Tn, int H, int W, int bands, float inv_div) {
  extern __shared__ float tile[];   // [3][VR_ROWS + 2][W + 2]
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int WP2 = W + 2, per_c = (VR_ROWS + 2) * WP2;
  const int band = blockIdx.x % bands;
  const int nt = blockIdx.x / bands;            // n * Tn + t
  const int t = nt % Tn, n = nt / Tn;
  const int h0 = band * VR_ROWS;
  __shared__ float lw[81];
  if (ty == 0 && tx < 27) { lw[tx] = lapw[tx]; lw[tx + 27] = lapw[tx + 27]; lw[tx + 54] = lapw[tx + 54]; }
  // tile fill: all loads of a row are issued before the first shared-memory store (the kernel is latency-bound otherwise)
  for (int r = ty; r < VR_ROWS + 2; r += 8) {
    const int hh = h0 + r - 1;
    const bool rin = (unsigned)hh < (unsigned)H;
    if (LAYOUT == 0) {
      const T* rp0 = video + ((((int64_t)n * 3) * Tn + t) * H + (rin ? hh : 0)) * W;
      const int64_t cstride = (int64_t)Tn * H * W;
      for (int col0 = 0; col0 < WP2; col0 += 128) {
        float vals[3][4];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int ww = col0 + tx + 32 * k - 1;
            vals[c][k] = (rin && (unsigned)ww < (unsigned)W) ? vr_norm<T>((float)rp0[c * cstride + ww]) : 0.f;
          }
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int col = col0 + tx + 32 * k;
            if (col < WP2) tile[c * per_c + r * WP2 + col] = vals[c][k];
          }
      }
    } else {
      const T* rp = video + (((int64_t)nt * H + (rin ? hh : 0)) * W) * 3;
      for (int e0 = 0; e0 < 3 * WP2; e0 += 256) {
        float vals[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int e = e0 + tx + 32 * k, col = e / 3, c = e - col * 3, ww = col - 1;
          vals[k] = (rin && e < 3 * WP2 && (unsigned)ww < (unsigned)W) ? vr_norm<T>((float)rp[ww * 3 + c]) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int e = e0 + tx + 32 * k, col = e / 3, c = e - col * 3;
          if (e < 3 * WP2) tile[c * per_c + r * WP2 + col] = vals[k];
        }
      }
    }
  }
  __syncthreads();
  const int h = h0 + ty;
  if (h >= H) return;
  // each thread produces strips of 4 consecutive pixels (two 16-byte units): the 3x6 neighbourhood and every laplacian
  // weight are read from shared memory once per strip instead of once per pixel
  const int64_t row_dst = (int64_t)(h & 1) * set_stride + uc_flat(g, n, t, h >> 1, 0) * 8 + 16;
  for (int p0 = 4 * tx; p0 < W; p0 += 128) {
    float acc[4][3];
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q][0] = acc[q][1] = acc[q][2] = 0.f;
    float ctr[4][3];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int ci = 0; ci < 3; ++ci) {
        float x[6];
        const float* trow = &tile[ci * per_c + (ty + kh) * WP2 + p0];
#pragma unroll
        for (int j = 0; j < 6; ++j) x[j] = (p0 + j < WP2) ? trow[j] : 0.f;   // tile columns p0 .. p0+5 <-> pixels p0-1 .. p0+4
        if (kh == 1) {
#pragma unroll
          for (int q = 0; q < 4; ++q) ctr[q][ci] = x[q + 1];
        }
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const int wi = ((kh * 3 + kw) * 3 + ci) * 3;
          const float w0 = lw[wi], w1 = lw[wi + 1], w2 = lw[wi + 2];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            acc[q][0] = fmaf(w0, x[q + kw], acc[q][0]);
            acc[q][1] = fmaf(w1, x[q + kw], acc[q][1]);
            acc[q][2] = fmaf(w2, x[q + kw], acc[q][2]);
          }
        }
      }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (p0 + 2 * u >= W) break;
      float px[8], lp[8];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const bool in = p0 + 2 * u + q < W;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          px[q * 4 + c] = in ? ctr[2 * u + q][c] : 0.f;
          lp[q * 4 + c] = in ? acc[2 * u + q][c] : 0.f;
        }
        px[q * 4 + 3] = 0.f;
        lp[q * 4 + 3] = 0.f;
      }
      *reinterpret_cast<uint4*>(xs + row_dst + (int64_t)(p0 + 2 * u) * 4) = pack8(px);
      *reinterpret_cast<uint4*>(xl + row_dst + (int64_t)(p0 + 2 * u) * 4) = pack8(lp);
    }
  }
}

// ---- bulk-copy (TMA engine) version --------------------------------------------------------------------------------------
// The register-heavy strip computation above leaves only two blocks per SM, too few to keep HBM busy with ordinary loads.
// Here the loads are asynchronous: persistent blocks walk (frame, band of VR2_ROWS rows) tiles, one elected thread streams
// the raw bytes of the next tiles (band + halo rows; one contiguous piece per channel plane, or one piece for interleaved
// layouts) into a VR2_STAGES-deep shared-memory ring with cp.async.bulk, completion on mbarriers; the 256 threads convert
// (uint8: /255) and compute from shared memory.  Column halos and rows outside the image are predicated, not staged.
// `starts` (optional, interleaved uint8 tracks): window n reads frames starts[n] .. starts[n]+T-1 of the track directly
// (the window builder of lsd_score_windows, video.py:552-556 + predictor.py:566-572, without materialising fp32 windows).
constexpr int VR2_ROWS = 16, VR2_STAGES = 3, VR2_THREADS = 256;
template <typename T> __device__ __forceinline__ void vr_load4(const T* p, float* o);
template <> __device__ __forceinline__ void vr_load4<float>(const float* p, float* o) {
  const float4 v = *reinterpret_cast<const float4*>(p);
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
template <> __device__ __forceinline__ void vr_load4<__half>(const __half* p, float* o) {
  const uint2 v = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
  o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
}
template <> __device__ __forceinline__ void vr_load4<__nv_bfloat16>(const __nv_bfloat16* p, float* o) {
  const uint2 v = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.x)), b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.y));
  o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
}
template <> __device__ __forceinline__ void vr_load4<uint8_t>(const uint8_t* p, float* o) {
  const uint32_t v = *reinterpret_cast<const uint32_t*>(p);
  o[0] = (float)(v & 0xffu) / 255.0f; o[1] = (float)((v >> 8) & 0xffu) / 255.0f;
  o[2] = (float)((v >> 16) & 0xffu) / 255.0f; o[3] = (float)(v >> 24) / 255.0f;
}
// uint8 through a 256-entry table of i / 255.0f (exactly the reference's astype(float32) / 255.0): twelve IEEE divisions per
// strip row made the uint8 variant ALU-bound and slower than the fp32 one although it reads a quarter of the bytes
template <typename T> __device__ __forceinline__ void vr_load4_lut(const T* p, float* o, const float*) { vr_load4<T>(p, o); }
// i / 255.0f for i in 0..255 without a division or a table: q = i * (1/255), one Newton step on the residual r = i - 255 q
// (both fused).  Bit-identical to the IEEE division for all 256 inputs (checked exhaustively against the division on the host,
// tests/test_host_logic.py, and by the uint8-vs-fp32 input equality test on the device).
__device__ __forceinline__ float vr_u8_norm(float x) {
  const float c = 1.0f / 255.0f;
  const float q = x * c;
  return fmaf(fmaf(-255.0f, q, x), c, q);
}
template <> __device__ __forceinline__ void vr_load4_lut<uint8_t>(const uint8_t* p, float* o, const float* lut) {
  const uint32_t v = *reinterpret_cast<const uint32_t*>(p);
  if (lut) { o[0] = lut[v & 0xffu]; o[1] = lut[(v >> 8) & 0xffu]; o[2] = lut[(v >> 16) & 0xffu]; o[3] = lut[v >> 24]; return; }
  o[0] = vr_u8_norm((float)(v & 0xffu)); o[1] = vr_u8_norm((float)((v >> 8) & 0xffu));
  o[2] = vr_u8_norm((float)((v >> 16) & 0xffu)); o[3] = vr_u8_norm((float)(v >> 24));
}
template <typename T> __device__ __forceinline__ float vr_norm_lut(T x, const float*) { return vr_norm<T>((float)x); }
template <> __device__ __forceinline__ float vr_norm_lut<uint8_t>(uint8_t x, const float* lut) { return lut ? lut[x] : vr_u8_norm((float)x); }

struct VrLapW { float w[81]; };   // [tap][ci][co], passed by value: the FFMAs take their weights from the constant bank
template <typename T, int LAYOUT>
__global__ void __launch_bounds__(VR2_THREADS, 3) video_rows_tma_kernel(const T* __restrict__ video, const int32_t* __restrict__ starts, int n_frames,
                                                                    const __grid_constant__ VrLapW LW, __nv_bfloat16* __restrict__ xs,
                                                                    __nv_bfloat16* __restrict__ xl, int64_t set_stride, UcGeom g, int Tn, int H, int W,
                                                                    int bands, int num_tiles) {
  extern __shared__ __align__(128) uint8_t vr_smem[];
  __shared__ uint64_t full_bar[VR2_STAGES];
  const float* lut = nullptr;   // (the table variant — 256 entries of i / 255.0f in shared memory — was bank-conflict-bound)
  const int tid = threadIdx.x;
  const int row_elems = LAYOUT == 0 ? W : 3 * W;                       // elements of one image row in one staged piece
  const int plane_elems = (VR2_ROWS + 2) * row_elems;                  // one staged piece (all rows of the band + halo)
  const uint32_t stage_bytes = (uint32_t)((LAYOUT == 0 ? 3 : 1) * plane_elems * (int)sizeof(T));
  const uint32_t stage_pitch = (stage_bytes + 127u) & ~127u;
  if (tid == 0) {
    for (int i = 0; i < VR2_STAGES; ++i) mbar_init(&full_bar[i], 1);
    fence_barrier_init();
  }
  __syncthreads();

  auto issue = [&](int k) {   // thread 0: stream tile k of this block into stage k % VR2_STAGES
    const int tile = blockIdx.x + k * gridDim.x;
    if (tile >= num_tiles) return;
    const int band = tile % bands, nt = tile / bands;
    const int h0 = band * VR2_ROWS;
    const int r_lo = h0 == 0 ? 1 : 0;                                    // first staged tile row (tile row r <-> image row h0-1+r)
    const int r_hi = min(VR2_ROWS + 2, H - h0 + 1);                      // one past the last staged tile row
    const uint32_t bytes = (uint32_t)((r_hi - r_lo) * row_elems * (int)sizeof(T));
    uint8_t* dst = vr_smem + (size_t)(k % VR2_STAGES) * stage_pitch + (size_t)r_lo * row_elems * sizeof(T);
    uint64_t* bar = &full_bar[k % VR2_STAGES];
    if (LAYOUT == 0) {
      const int n = nt / Tn, t = nt - n * Tn;
      mbar_arrive_expect_tx(bar, 3u * bytes);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const T* src = video + ((((int64_t)n * 3 + c) * Tn + t) * H + (h0 - 1 + r_lo)) * W;
        bulk_g2s(dst + (size_t)c * plane_elems * sizeof(T), src, bytes, bar);
      }
    } else {
      int64_t frame = nt;
      if (starts) {
        const int n = nt / Tn, t = nt - n * Tn;
        int f = starts[n] + t;
        frame = f < 0 ? 0 : (f >= n_frames ? n_frames - 1 : f);
      }
      mbar_arrive_expect_tx(bar, bytes);
      bulk_g2s(dst, video + (frame * H + (h0 - 1 + r_lo)) * (int64_t)row_elems, bytes, bar);
    }
  };
  if (tid == 0)
    for (int k = 0; k < VR2_STAGES - 1; ++k) issue(k);

  const int nstrips = W >> 2;
  const int ntasks = VR2_ROWS * nstrips;
  for (int k = 0;; ++k) {
    const int tile = blockIdx.x + k * gridDim.x;
    if (tile >= num_tiles) break;
    if (tid == 0) issue(k + VR2_STAGES - 1);      // its stage was drained before the barrier that ended iteration k-1
    mbar_wait(&full_bar[k % VR2_STAGES], (uint32_t)(k / VR2_STAGES) & 1u);
    const T* st = reinterpret_cast<const T*>(vr_smem + (size_t)(k % VR2_STAGES) * stage_pitch);
    const int band = tile % bands, nt = tile / bands;
    const int n = nt / Tn, t = nt - n * Tn;
    const int h0 = band * VR2_ROWS;
    for (int task = tid; task < ntasks; task += VR2_THREADS) {
      const int ty = task / nstrips, p0 = (task - ty * nstrips) << 2;
      const int h = h0 + ty;
      if (h >= H) break;
      float acc[4][3], ctr[4][3];
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[q][0] = acc[q][1] = acc[q][2] = 0.f;
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        const int hh = h - 1 + kh;
        float x[3][6];   // channel, pixels p0-1 .. p0+4
        if ((unsigned)hh < (unsigned)H) {
          const T* trow = st + (size_t)(ty + kh) * row_elems;
          if (LAYOUT == 0) {
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) {
              const T* pr = trow + (size_t)ci * plane_elems + p0;
              vr_load4_lut<T>(pr, &x[ci][1], lut);
              x[ci][0] = p0 > 0 ? vr_norm_lut<T>(pr[-1], lut) : 0.f;
              x[ci][5] = p0 + 4 < W ? vr_norm_lut<T>(pr[4], lut) : 0.f;
            }
          } else {
            const T* pr = trow + 3 * p0;
            float e[12];
            vr_load4_lut<T>(pr, e, lut); vr_load4_lut<T>(pr + 4, e + 4, lut); vr_load4_lut<T>(pr + 8, e + 8, lut);
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
              for (int ci = 0; ci < 3; ++ci) x[ci][q + 1] = e[q * 3 + ci];
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) {
              x[ci][0] = p0 > 0 ? vr_norm_lut<T>(pr[ci - 3], lut) : 0.f;
              x[ci][5] = p0 + 4 < W ? vr_norm_lut<T>(pr[12 + ci], lut) : 0.f;
            }
          }
        } else {
#pragma unroll
          for (int ci = 0; ci < 3; ++ci)
#pragma unroll
            for (int j = 0; j < 6; ++j) x[ci][j] = 0.f;
        }
        if (kh == 1) {
#pragma unroll
          for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int ci = 0; ci < 3; ++ci) ctr[q][ci] = x[ci][q + 1];
        }
#pragma unroll
        for (int ci = 0; ci < 3; ++ci)
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            const int wi = ((kh * 3 + kw) * 3 + ci) * 3;
            const float w0 = LW.w[wi], w1 = LW.w[wi + 1], w2 = LW.w[wi + 2];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              acc[q][0] = fmaf(w0, x[ci][q + kw], acc[q][0]);
              acc[q][1] = fmaf(w1, x[ci][q + kw], acc[q][1]);
              acc[q][2] = fmaf(w2, x[ci][q + kw], acc[q][2]);
            }
          }
      }
      const int64_t dst = (int64_t)(h & 1) * set_stride + uc_flat(g, n, t, h >> 1, 0) * 8 + 16 + (int64_t)p0 * 4;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        float px[8], lp[8];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
#pragma unroll
          for (int c = 0; c < 3; ++c) { px[q * 4 + c] = ctr[2 * u + q][c]; lp[q * 4 + c] = acc[2 * u + q][c]; }
          px[q * 4 + 3] = 0.f; lp[q * 4 + 3] = 0.f;
        }
        *reinterpret_cast<uint4*>(xs + dst + u * 8) = pack8(px);
        *reinterpret_cast<uint4*>(xl + dst + u * 8) = pack8(lp);
      }
    }
    __syncthreads();   // every thread is done with this stage before it is refilled (issue(k + STAGES) at iteration k + 1)
  }
}

cudaError_t video_rows_device_init() {
  cudaError_t e = cudaSuccess;
#define VRA(TT, LL) if (e == cudaSuccess) e = cudaFuncSetAttribute(video_rows_tma_kernel<TT, LL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)
  VRA(float, 0); VRA(__half, 0); VRA(__nv_bfloat16, 0); VRA(uint8_t, 0);
  VRA(float, 1); VRA(__half, 1); VRA(__nv_bfloat16, 1); VRA(uint8_t, 1);
#undef VRA
  return e;
}

bool video_rows_bulk_ok(const void* video, int dtype, int layout, int W) {
  const size_t esz = dtype == 0 ? 4 : (dtype == 3 ? 1 : 2);
  const size_t row_bytes = (size_t)W * esz * (layout == 0 ? 1 : 3);
  const size_t stage = (((layout == 0 ? 3 : 1) * (size_t)(VR2_ROWS + 2) * row_bytes) + 127) & ~size_t(127);
  return (W % 4 == 0) && (row_bytes % 16 == 0) && (reinterpret_cast<uintptr_t>(video) % 16 == 0) && stage * VR2_STAGES <= 96 * 1024;
}

void launch_video_rows(const void* video, int dtype, int layout, const float* lapw, const float* lapw_host, __nv_bfloat16* xs, __nv_bfloat16* xl,
                       int64_t set_stride, UcGeom g, int H, int W, cudaStream_t s, int num_sms, const int32_t* starts, int n_frames) {
  const size_t esz = dtype == 0 ? 4 : (dtype == 3 ? 1 : 2);
  const size_t row_bytes = (size_t)W * esz * (layout == 0 ? 1 : 3);
  const size_t stage = (((layout == 0 ? 3 : 1) * (size_t)(VR2_ROWS + 2) * row_bytes) + 127) & ~size_t(127);
  if (video_rows_bulk_ok(video, dtype, layout, W)) {
    const int bands = (H + VR2_ROWS - 1) / VR2_ROWS;
    const int64_t tiles = (int64_t)g.N * g.T * bands;
    if (tiles == 0) return;
    const size_t smem = stage * VR2_STAGES;
    VrLapW lw;
    memcpy(lw.w, lapw_host, sizeof(lw.w));
    const int64_t per_sm = stage * VR2_STAGES * 3 <= 200 * 1024 ? 3 : 2;   // 80 registers x 256 threads, <= 62 KB of stages: three resident blocks per SM
    const unsigned grid = (unsigned)std::min<int64_t>(tiles, per_sm * num_sms);
#define VRT(TT, LL)                                                                                                             \
  do {                                                                                                                          \
    video_rows_tma_kernel<TT, LL><<<grid, VR2_THREADS, smem, s>>>(reinterpret_cast<const TT*>(video), starts, n_frames, lw, xs, xl,    \
                                                                  set_stride, g, g.T, H, W, bands, (int)tiles);               \
  } while (0)
    if (layout == 0) {
      if (dtype == 0) VRT(float, 0); else if (dtype == 1) VRT(__half, 0); else if (dtype == 2) VRT(__nv_bfloat16, 0); else VRT(uint8_t, 0);
    } else {
      if (dtype == 0) VRT(float, 1); else if (dtype == 1) VRT(__half, 1); else if (dtype == 2) VRT(__nv_bfloat16, 1); else VRT(uint8_t, 1);
    }
#undef VRT
    count_launch();
    return;
  }
  // fallback (unaligned rows / odd widths): direct loads; a start table is not supported here (the caller gathers first)
  const int bands = (H + VR_ROWS - 1) / VR_ROWS;
  const int64_t blocks = (int64_t)g.N * g.T * bands;
  if (blocks == 0) return;
  const size_t smem = (size_t)3 * (VR_ROWS + 2) * (W + 2) * sizeof(float);
#define VR(TT, LL, DIV) video_rows_kernel<TT, LL><<<(unsigned)blocks, dim3(32, 8), smem, s>>>(reinterpret_cast<const TT*>(video), lapw, xs, xl, set_stride, g, g.T, H, W, bands, 1.0f / (DIV))
  if (layout == 0) {
    if (dtype == 0) VR(float, 0, 1.0f); else if (dtype == 1) VR(__half, 0, 1.0f); else if (dtype == 2) VR(__nv_bfloat16, 0, 1.0f); else VR(uint8_t, 0, 255.0f);
  } else {
    if (dtype == 0) VR(float, 1, 1.0f); else if (dtype == 1) VR(__half, 1, 1.0f); else if (dtype == 2) VR(__nv_bfloat16, 1, 1.0f); else VR(uint8_t, 1, 255.0f);
  }
#undef VR
  count_launch();
}

// Generalised deterministic mean (see token_kernels.cuh): fp32 rows and/or planar bf16 rows out.
__global__ void planar_mean2_kernel(const __nv_bfloat16* __restrict__ x, int64_t plane_stride, UcGeom g, float* __restrict__ y32, int ld,
                                    int mode, PlanarOut po, const __nv_bfloat16* __restrict__ xlo) {
  __shared__ float part[256][9];
  const int row = blockIdx.x, chunk = blockIdx.y, tid = threadIdx.x;
  const int count = mode == 1 ? g.T * g.H * g.W : (mode == 0 ? g.H * g.W : g.H);
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  auto add = [&](int64_t pos) {
    float f[8];
    const int64_t src = (int64_t)chunk * plane_stride + pos * 8;
    unpack8(*reinterpret_cast<const uint4*>(x + src), f);
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] += f[e];
    if (xlo) {
      unpack8(*reinterpret_cast<const uint4*>(xlo + src), f);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += f[e];
    }
  };
  if (mode == 2) {
    const int n = row / g.W, w = row % g.W;
    for (int i = tid; i < count; i += blockDim.x) add(uc_flat(g, n, 0, i, w));
  } else {
    // one image row (t, h) per warp and step, lanes along w: the positions of a row are contiguous, and the per-element
    // divisions of a flat index (four per 16-byte load) no longer bound the kernel
    const int n = mode == 1 ? row : row / g.T, t0 = mode == 1 ? 0 : row % g.T;
    const int n_rows = (mode == 1 ? g.T : 1) * g.H;
    const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    if (g.W <= 32 && !xlo) {
      // rows of at most one warp width: four rows in flight per warp (the loads are issued before the first dependent add; the
      // summation order is the sequential one)
      const bool act = lane < g.W;
      const __nv_bfloat16* xc = x + (int64_t)chunk * plane_stride;
      int rr = warp;
      for (; rr + 3 * nwarps < n_rows; rr += 4 * nwarps) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int r = rr + u * nwarps, tt = r / g.H, h = r - tt * g.H;
          v[u] = act ? *reinterpret_cast<const uint4*>(xc + (uc_flat(g, n, t0 + tt, h, 0) + lane) * 8) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          float f[8];
          unpack8(v[u], f);
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[e] += f[e];
        }
      }
      for (; rr < n_rows; rr += nwarps) {
        const int tt = rr / g.H, h = rr - tt * g.H;
        if (act) add(uc_flat(g, n, t0 + tt, h, 0) + lane);
      }
    } else
    for (int rr = warp; rr < n_rows; rr += nwarps) {
      const int tt = rr / g.H, h = rr - tt * g.H;
      const int64_t base = uc_flat(g, n, t0 + tt, h, 0);
      for (int w = lane; w < g.W; w += 32) add(base + w);
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) part[tid][e] = acc[e];
  __syncthreads();
  for (int sft = blockDim.x >> 1; sft > 0; sft >>= 1) {
    if (tid < sft) {
#pragma unroll
      for (int e = 0; e < 8; ++e) part[tid][e] += part[tid + sft][e];
    }
    __syncthreads();
  }
  if (tid < 8) {
    const float m = part[0][tid] / (float)count;
    if (y32) y32[(int64_t)row * ld + chunk * 8 + tid] = m;
    if (po.y) {
      const int64_t pos = po.grp > 0 ? ((int64_t)row / po.grp) * po.grp_stride + (row % po.grp) + po.off : (int64_t)row + po.off;
      const __nv_bfloat16 hi = __float2bfloat16_rn(m);
      po.y[(int64_t)chunk * po.plane_stride + pos * 8 + tid] = hi;
      if (po.ylo) po.ylo[(int64_t)chunk * po.plane_stride + pos * 8 + tid] = __float2bfloat16_rn(m - __bfloat162float(hi));
    }
  }
}
// Short means (<= 32 positions: the 3x3 spatial mean of the visual tokens, the mean over F' = 3 of the audio tokens): one
// THREAD per (row, 8-channel chunk) summing serially — the block-per-row tree above launched 65k one-warp blocks for 9 values.
__global__ void __launch_bounds__(256) planar_mean2_small_kernel(const __nv_bfloat16* __restrict__ x, int64_t plane_stride, UcGeom g,
                                                                 float* __restrict__ y32, int ld, int mode, PlanarOut po,
                                                                 const __nv_bfloat16* __restrict__ xlo, int rows, int nchunks) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * nchunks) return;
  const int chunk = i / rows, row = i - chunk * rows;      // consecutive threads -> consecutive rows of one plane
  const int count = mode == 0 ? g.H * g.W : g.H;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int k = 0; k < count; ++k) {
    int n, t, h, w;
    if (mode == 2) { n = row / g.W; w = row - n * g.W; t = 0; h = k; }
    else { n = row / g.T; t = row - n * g.T; h = k / g.W; w = k - h * g.W; }
    const int64_t off = (int64_t)chunk * plane_stride + uc_flat(g, n, t, h, w) * 8;
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(x + off), f);
    if (xlo) {
      float fl[8];
      unpack8(*reinterpret_cast<const uint4*>(xlo + off), fl);
#pragma unroll
      for (int e = 0; e < 8; ++e) f[e] += fl[e];
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] += f[e];
  }
  float m[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) m[e] = acc[e] / (float)count;
  if (y32) {
    float4* o = reinterpret_cast<float4*>(y32 + (int64_t)row * ld + chunk * 8);
    o[0] = make_float4(m[0], m[1], m[2], m[3]);
    o[1] = make_float4(m[4], m[5], m[6], m[7]);
  }
  if (po.y) {
    const int64_t pos = po.grp > 0 ? ((int64_t)row / po.grp) * po.grp_stride + (row % po.grp) + po.off : (int64_t)row + po.off;
    const uint4 hi4 = pack8(m);
    *reinterpret_cast<uint4*>(po.y + (int64_t)chunk * po.plane_stride + pos * 8) = hi4;
    if (po.ylo) {
      float hf[8], lo[8];
      unpack8(hi4, hf);
#pragma unroll
      for (int e = 0; e < 8; ++e) lo[e] = m[e] - hf[e];
      *reinterpret_cast<uint4*>(po.ylo + (int64_t)chunk * po.plane_stride + pos * 8) = pack8(lo);
    }
  }
}

void launch_planar_mean2(const __nv_bfloat16* x, int64_t plane_stride, UcGeom g, int C, float* y32, int ld, int mode, PlanarOut po, cudaStream_t s,
                         const __nv_bfloat16* xlo) {
  const int rows = mode == 1 ? g.N : (mode == 0 ? g.N * g.T : g.N * g.W);
  if (rows == 0) return;
  const int count = mode == 1 ? g.T * g.H * g.W : (mode == 0 ? g.H * g.W : g.H);
  if (mode != 1 && count <= 32 && (ld % 4) == 0 && (!y32 || reinterpret_cast<uintptr_t>(y32) % 16 == 0)) {
    const int total = rows * (C / 8);
    planar_mean2_small_kernel<<<(total + 255) / 256, 256, 0, s>>>(x, plane_stride, g, y32, ld, mode, po, xlo, rows, C / 8);
    count_launch();
    return;
  }
  int threads = 32;
  while (threads < 256 && threads < count) threads <<= 1;
  planar_mean2_kernel<<<dim3(rows, C / 8), threads, 0, s>>>(x, plane_stride, g, y32, ld, mode, po, xlo);
  count_launch();
}

}  // namespace lsd
