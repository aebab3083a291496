// Fused front of the token path (tok_front.cu): everything between the cross-attention input projections and the first
// transformer layer in ONE launch — the two cross-modal attention directions with their output projections and residuals, the
// gated fusion (Linear 512->256, GELU, Linear 256->1, sigmoid, blend, Linear 256->256, ReLU: app/models/fusion_module.py:67-87),
// the three multi-scale Conv1d branches (k = 3, 5, 7; BN folded; GELU), their concatenation through pre_scale_proj, the
// residual and the CLS row (app/models/temporal.py:95-107).  Replaces 12 launches of the layer-by-layer chain.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace lsd {

constexpr int TFR_STAGE_BYTES = 16384;   // every weight-ring stage: 2 K16 steps of a 256-column block, packed [k16][2 planes][256][8] fp16
// Weight stream, in the order the MMA warp consumes it (K16 steps; all blocks are 256 columns wide):
//   out_proj of v2a, head pairs 0..3 (4 each) | out_proj of a2v (4 x 4) | gate.0 (32) | fuse.0 (16) |
//   branch_k3 (3 taps x 16) | pre_scale_proj[:, 0:256] (16) | branch_k5 (5 x 16) | pre_scale_proj[:, 256:512] (16) |
//   branch_k7 (7 x 16) | pre_scale_proj[:, 512:768] (16)
constexpr int TFR_K16_TOTAL = 16 + 16 + 32 + 16 + 48 + 16 + 80 + 16 + 112 + 16;
constexpr int TFR_N_STAGES = TFR_K16_TOTAL / 2;
// fp32 vector block: [bo_v2a | bo_a2v | gate0 bias | gate2 weight | gate2 bias (1, padded to 64) | fuse bias | BN shift k3 | k5 | k7 |
//                     pre_scale bias | cls token]
enum { TFR_V_BO0 = 0, TFR_V_BO1 = 256, TFR_V_BG0 = 512, TFR_V_WG2 = 768, TFR_V_BG2 = 1024, TFR_V_BF = 1088, TFR_V_SH3 = 1344, TFR_V_SH5 = 1600,
       TFR_V_SH7 = 1856, TFR_V_BP = 2112, TFR_V_CLS = 2368, TFR_V_TOTAL = 2624 };

struct TokFrontP {
  int ld_p, ld_e;       // row strides (floats) of pv / pa and of v_emb / a_int
  const float* pv;      // [B*T][768] fp32: [Q of v2a | K of a2v | V of a2v] of the visual tokens (in-projection output, bias included)
  const float* pa;      // [B*T][768] fp32: [Q of a2v | K of v2a | V of v2a] of the interpolated audio tokens
  const float* v_emb;   // [B*T][256] fp32 residual of v2a
  const float* a_int;   // [B*T][256] fp32 residual of a2v (audio tokens interpolated to T)
  float* gi;            // [B*T][512] fp32 scratch: [v_out | a_out]
  float* fused;         // [B*T][256] fp32 out: CrossModalAttention.forward
  float* tok;           // [B][T+1][256] fp32 out: row 0 = cls token, rows 1..T = fused + pre_scale_proj(cat(branches))
  const __half* w;      // packed weight stream (TFR_N_STAGES stages)
  const float* vec;     // TFR_V_TOTAL floats
  void* dbg;            // optional (LSD_TOKF_TRACE): 256 x int64 phase timestamps of CTA 0 (MMA warp: [0,128), compute warp 0: [128,256))
  int B, T, SL, G, KW;  // windows, tokens per window, row slot per window (32 or 64; >= T + 3), windows per CTA, keys per window (16-multiple)
  int K;                // visual row group: window w reads the visual rows (pv, v_emb) of window w / K (K audio variants share one
                        // visual window, lsd_forward_audio_variants); 1 = every window has its own visual rows
};

cudaError_t tok_front_device_init();
bool tok_front_supported(int T);
void tok_front_geometry(int T, int& SL, int& G, int& KW);
void launch_tok_front(const TokFrontP& p, cudaStream_t s);

}  // namespace lsd
