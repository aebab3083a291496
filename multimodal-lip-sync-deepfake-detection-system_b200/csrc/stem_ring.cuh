// "Temporal ring" stem convolution (stem_ring.cu): Conv3d(3 -> 64, 3x7x7, stride (1,2,2)) + BN + ReLU of
// app/models/visual_encoder.py:113-125 with the three temporal taps as three 64-column blocks of ONE N = 192 tcgen05 MMA.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "umma_conv.cuh"

namespace lsd {

constexpr int SR_TAPS = 7;                 // (parity set, dh) pairs = the 7 kernel rows
constexpr int SR_WBLOCK = 2 * 192 * 16;    // bytes of one (tap, K chunk) weight block: [2 K halves][192 columns][8 bf16]
constexpr int SR_WBYTES = SR_TAPS * 2 * SR_WBLOCK;

// One step of one accumulator slot: the input slab t_in of one 128-position column chunk.  The output slab that completes with the
// step is the same chunk one slab earlier (in_pos - SL).
struct alignas(8) SrStep {
  int32_t in_pos;     // flat position (geometry g) of the chunk's first position in the INPUT slab of this step
  uint32_t flags;     // bit 0: active, bit 1: first step of a segment (all three accumulator blocks start from the bias),
                      // bit 2: the completed block is stored, bits 8-15: positions of the chunk that lie inside the slab (<= 128)
};
constexpr uint32_t SR_ACTIVE = 1u, SR_FIRST = 2u, SR_STORE = 4u;

struct StemRingP {
  const __nv_bfloat16* xs[2];   // pixel rows, h-parity plane sets (position 0 of each)
  const __nv_bfloat16* w;       // packed weights, SR_WBYTES: [tap][K chunk][K half][dt block j: 0..2][64][8]
  const float* bias;            // 64 (BN shift)
  __nv_bfloat16* y;             // planar destination, plane 0 / position 0, geometry g
  int64_t y_plane_stride;
  UcGeom g;
  const SrStep* steps;          // [2 * gridDim.x slots][nsteps]; every CTA copies its two rows into shared memory first
  int nsteps;
  int skip;                     // timing experiments (LSD_SR_SKIP, garbage results): bit 0 epilogue without loads / stores, bit 1 no wrap MMAs
                                // (D region pinned to block 0), bit 2 only two of the seven taps
  long long* dbg;               // optional (LSD_SR_TRACE): CTA 0 writes clock64 stamps of steps 16..47: [role 0..3][32 steps][2]
  int ntap[2];                  // taps per parity set
  int rel[2][4];                // tap offsets (positions) relative to the region start of their set
  int start[2];                 // region start relative to the chunk's first position
  int units[2];                 // region length in positions (16 B each)
  int nst;                      // ring stages of the pixel-row regions (6; fewer when a long step table needs the shared memory)
};

cudaError_t stem_ring_device_init();
size_t stem_ring_smem_bytes(const StemRingP& p);
void launch_stem_ring(const StemRingP& p, int grid, cudaStream_t s);

}  // namespace lsd
