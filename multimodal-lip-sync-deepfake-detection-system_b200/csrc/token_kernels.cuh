// Token-path kernels of the bf16 route (token_kernels.cu): fp32 math, planar bf16 hand-off to the tcgen05 GEMMs.
#pragma once
#include "lsd_kernels.h"
#include "umma_conv.cuh"

namespace lsd {

// Destination of a row-wise result in padded planar bf16: position(row) = (row/grp)*grp_stride + row%grp + off
// (grp == 0: position = row + off); element (row, c) lives at y[(c/8)*plane_stride + position*8 + c%8].
struct PlanarOut {
  __nv_bfloat16* y;
  __nv_bfloat16* ylo;   // optional: receives bf16(v - bf16(v)) at the same position (split-bf16 GEMM operands)
  int64_t plane_stride;
  int grp, grp_stride, off;
};

struct HeadW {  // fp32 arena pointers, weights as [Cin][Cout]
  const float *w0, *b0, *w2, *b2, *wc, *bc, *lng, *lnb, *wo, *bo;
};

void launch_layernorm_p(const float* x, int64_t x_ld, const float* g, const float* b, int rows, int D, PlanarOut o, cudaStream_t s);
void launch_mha_core_p(const float* q, int q_ld, const float* k, int k_ld, const float* v, int v_ld, int N, int Tq, int Tk, int heads,
                       PlanarOut o, cudaStream_t s);
void launch_gate_blend_p(const float* h, const float* w2, const float* b2, const float* v, int v_ld, const float* a, int a_ld, int rows,
                         int D, PlanarOut o, cudaStream_t s);
void launch_lerp_tokens_p(const float* x, float* y, int N, int Tin, int Tout, int D, PlanarOut o, cudaStream_t s);
void launch_audio_rows(const void* audio, int dtype, __nv_bfloat16* y, int64_t set_stride, UcGeom g, int F, int Ta, cudaStream_t s);
// K: windows n = b*K + k read the artifact features comb[b] (audio variants of one video); 1 = one comb row per window
void launch_head(const float* cls, int64_t cls_ld, const float* comb, const HeadW& w, float* logits, int B, cudaStream_t s, int K = 1);
// mean of a planar tensor -> fp32 rows (y32, may be null) and/or planar bf16 rows (po.y, may be null)
//   mode 0: one row per (n,t), mean over H*W;  mode 1: one row per window, mean over T*H*W;  mode 2: one row per (n,w), mean over H (T == 1)
void launch_planar_mean2(const __nv_bfloat16* x, int64_t plane_stride, UcGeom g, int C, float* y32, int ld, int mode, PlanarOut po, cudaStream_t s,
                         const __nv_bfloat16* xlo = nullptr);

}  // namespace lsd
