// Parameter block of the tcgen05 "flat shift-GEMM" convolution kernel (umma_conv.cu) and the planar-layout glue.
//
// Activation layout of the bf16 path ("padded planar"): a tensor (N, T, H, W, C) is stored as C/8 planes; one plane
// holds, for every *padded flat position*
//     P = ((n*(T+1) + t + 1) * (H+1) + (h+1)) * (W+1) + (w+1)
// the 8 channels of that position (16 bytes).  Slab 0 of every window, row 0 of every slab and column 0 of every row
// are zero (one shared pad between neighbours), so a 3x3x3 / pad-1 convolution is a pure shift in P:
//     out[P] = sum_taps W_tap . in[P + (kt-1)*SL + (kh-1)*RW + (kw-1)],   RW = W+1,  SL = (H+1)*(W+1)
// and 8 consecutive positions of one channel-chunk are exactly one 8x16B UMMA core matrix (K-major, no swizzle).
// Stride-2 consumers read a "parity-split" tensor: 4 plane sets (h&1, w&1), each in the half-resolution geometry.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace lsd {

constexpr int UC_MAX_BANDS = 16;
constexpr int UC_MAX_TAPS = 12;
constexpr int UC_MAX_GROUPS = 6;

struct UcBand {
  const __nv_bfloat16* base;  // plane 0, position 0 of the plane set this band reads
  int64_t plane_stride;       // elements between consecutive 8-channel planes
  int64_t chunk_stride;       // elements added per k16 chunk: 2*plane_stride (planar) or 16 (Toeplitz pixel rows)
  int start;                  // flat shift of the band's first position relative to the tile's first position
  int len_extra;              // band length = tile positions + len_extra
  int ntaps;
  int tap_begin;              // index of the band's first tap inside its group's packed weights
  int toeplitz;               // 1: K runs along the pixel row itself (LBO = 16 B, one region), see bf16_path.cu (stem / hf front)
  int rel[UC_MAX_TAPS];       // tap shift relative to the band start (positions)
};

struct UcGroup {              // taps that share one K extent (main conv; optional fused 1x1 downsample)
  int band_begin, band_end;
  int k16;                    // Cin / 16
  int taps_total;
  int64_t w_off;              // element offset of the group's packed weights
  int64_t slice_stride;       // elements between consecutive Cout slices (grid.y) of the packed weights
};

// bf16 planar output modes (an fp32 row output can be produced in addition to, or instead of, the planar one)
// UC_Y_FOLD: "folded" destination (small maps, see UcFoldSlice): plane set h*ymap_W + w, position = frame row uc_flat(g2, n, t, 0, 0).
// UC_Y_MAP: plain padded planar destination in geometry g2 written at (n, t, h, w) — a folded conv's output back in the map layout.
enum UcOut { UC_Y_NONE = 0, UC_Y_PLAIN = 1, UC_Y_PARITY = 2, UC_Y_PARITY_H = 3, UC_Y_FOLD = 5, UC_Y_MAP = 6 };

// Folded small-map convolution ("frames as rows").  A map of H x W x C per frame is stored as H*W plane sets (one per spatial
// position) in the row geometry make_geom_ex(N, T, 1, 1, 1, 0, 0, 0, 0): position = frame row n*(T+1) + t + 1, with the shared
// zero row of every window.  A 3x3x3 / pad-1 convolution is then, per output position p, a 3-tap temporal convolution (row
// shifts -1 / 0 / +1) summed over the input positions q that p's 3x3 stencil reaches IN BOUNDS: no multiply reads padding,
// and no position outside the map is computed.  Each column slice (grid.y) is one (output position, Cout slice) with its own
// stage program: one band per in-bounds q (three temporal taps, A from plane set q), then the fused 1x1 downsample band.
constexpr int UC_MAX_FSLICES = 96;
struct UcFoldSlice {
  uint16_t prog_off, nst;     // the slice's stage program: prog[prog_off .. prog_off + nst)
  uint8_t h, w;               // output position in the map
  uint8_t col, pad_;          // Cout slice (columns col*Cout ..)
};

// Padded flat geometry:  P = ((n*TS + t + ot)*HP + h + oh)*RW + w + ow,  SL = HP*RW.
// Standard activation geometry: one shared zero slab / row / column (TS=T+1, ot=1, HP=H+1, oh=1, RW=W+1, ow=1).
struct UcGeom {
  int N, T, H, W;
  int TS, ot, HP, oh, RW, ow, SL;
  int64_t P_total;
  // division by SL / RW / TS as multiply + shift (numerators < 2^31): q = (n * m) >> (31 + s), see uc_magic
  uint32_t mSL, mRW, mTS;
  int sSL, sRW, sTS;
};

// Round-up magic number for dividing numerators n < 2^31 by d >= 1: s = ceil(log2 d), m = floor(2^(31+s) / d) + 1 < 2^32;
// m*d = 2^(31+s) + e with 0 < e <= d <= 2^s, so n*e < 2^(31+s) and floor(n*m / 2^(31+s)) == floor(n / d).
inline void uc_magic(uint32_t d, uint32_t& m, int& s) {
  s = 0;
  while (((uint64_t)1 << s) < d) ++s;
  m = (uint32_t)((((uint64_t)1 << (31 + s)) / d) + 1);
}

// One ring stage of a tile, as the producers and MMA issuers consume it ("stage program").  The sequence of stages
// (group, K-chunk block, band) is identical for every tile — only the tile's first position shifts the A sources — so the host
// expands it once per (layer, shapes, workspace), keeps it in device memory (lsd_handle::prog_*) and every CTA copies it into
// shared memory in its prologue.  Computing the same operands in the kernel from the parameter block cost ~150 dependent
// instructions (indexed constant loads, 64-bit multiplies) = ~1200 cycles per stage for the single issuing warp, more than the
// MMA time of a stage for every layer with few taps per stage (token GEMMs, audio encoder, 256-column tiles).
struct alignas(16) UcStageDesc {
  uint64_t a_src;            // global byte address of the stage's first A piece for tile position 0
  uint64_t w_src;            // global byte address of the stage's first weight piece, Cout slice 0
  uint64_t chunk_stride_b;   // bytes between consecutive K-chunk pairs of planes
  uint64_t plane_stride_b;   // bytes between the two 8-channel planes of a K chunk
  uint64_t w_slice_stride_b; // bytes between consecutive Cout slices of the packed weights
  uint32_t bytesA;           // bytes of one A piece
  uint32_t w_copy_bytes;     // bytes of one weight copy
  uint32_t w_dst_step;       // shared-memory distance between weight pieces
  uint32_t w_src_step;       // global distance between the weight pieces of consecutive K chunks
  uint32_t tx_bytes;         // bytes the stage's full barrier expects
  uint32_t counts;           // n_a | n_w << 8 | band index << 16 | K chunks in this stage << 24
};
static_assert(sizeof(UcStageDesc) == 64, "UcStageDesc must be 64 bytes");

struct UmmaConvP {
  const __nv_bfloat16* w;     // packed: [group][Cout slice][k16 chunk][tap][2 k-chunks][Cout][8]
  const float* bias;          // all slices (BN shift + folded conv bias; BN scale is folded into w)
  const __nv_bfloat16* res;   // optional bf16 residual, plain layout in the output geometry
  const __nv_bfloat16* res_lo; // optional low part of the residual (split-bf16 activations)
  int64_t res_plane_stride;
  const float* res32;         // optional fp32 residual rows: res32[(outer*W + w) * res32_ld + channel]
  int res32_ld;
  __nv_bfloat16* y;           // planar destination (position 0 of plane 0 [of set 0]); y_mode selects the layout
  __nv_bfloat16* ylo;         // optional second planar destination receiving bf16(v - bf16(v)) (split-bf16 operands of the
                              //   token-path GEMMs: x ~ hi + lo keeps ~16 mantissa bits through the tensor cores)
  int64_t y_plane_stride, y_set_stride;
  int y_mode;
  float* y32;                 // optional fp32 rows: y32[(outer*y32_outer_stride + w + y32_row_off) * y32_ld + channel],
  int y32_ld;                 //   outer = (n*T + t)*H + h  (valid positions only)
  int y32_outer_stride, y32_row_off;
  int act;
  int Cout;                   // columns per CTA (one slice); grid.y = number of slices
  int MT, stages, ngroups, nbands;
  int issuers;                // MMA-issuing warps (1, 2 or 4; divides MT): each issues MT / issuers M-tiles per tap
  int nbuf;                   // TMEM accumulator buffers: 2 = epilogue overlaps the next tile, 1 = all 512 columns for one tile
  long long* dbg;             // optional: CTA (0,0) writes clock64 phase timestamps (debug builds of the bench only)
  const UcStageDesc* prog;    // device memory: the stage program (nst_tile entries)
  int nst_tile;               // ring stages per tile (sum over groups of ceil(k16 / kpack) * bands): length of the stage program
  int skip;                   // debug (LSD_UMMA_SKIP): bit 0 = no A copies, bit 1 = no W copies — timing experiments only
  int kpack;                  // k16 chunks per pipeline stage (small-K-step layers amortise the mbarrier round trip)
  uint32_t a_stage_bytes, w_stage_bytes, tmem_cols;
  int cta2;                   // 1: CTA pairs (cluster of 2, tcgen05 cta_group::2): the packed weights hold two column halves as slices
  UcGeom g;                   // output geometry (== input geometry of every band)
  UcGeom g2;                  // UC_Y_PARITY* / UC_Y_FOLD / UC_Y_MAP: destination geometry (of each plane set)
  UcGroup groups[UC_MAX_GROUPS];
  UcBand bands[UC_MAX_BANDS];
  int ymap_W;                 // UC_Y_FOLD: width of the map whose positions are the destination's plane sets
  int fold;                   // 1: folded conv — grid.y walks fslice[]; the stage program is per slice, one tile per CTA
  UcFoldSlice fslice[UC_MAX_FSLICES];
};

size_t umma_conv_smem_bytes(const UmmaConvP& p);
int umma_conv_stage_desc_bytes();
size_t umma_conv_extra_smem_bytes(const UmmaConvP& p);   // behind the stage program: bias operand tiles (lean epilogue)
// host: expand the stage program of a launch (same arithmetic the kernel used to do per stage)
void umma_conv_build_program(const UmmaConvP& p, UcStageDesc* out);
// host: one stage (K chunks c0 .. c0 + nc of band bd, whose index in p.bands is `band`); col >= 0: the Cout slice is baked into
// the weight address (folded convs, whose grid.y is not the Cout slice)
UcStageDesc umma_conv_stage(const UmmaConvP& p, const UcGroup& g, const UcBand& bd, int band, int c0, int col = -1);
// nullptr if the kernel supports this parameter block, else the reason (callers turn it into an error code instead of launching)
const char* umma_conv_config_error(const UmmaConvP& p);
void launch_umma_conv(const UmmaConvP& p, int n_slices, cudaStream_t s, int num_sms, int max_ctas = 0);
// per-device one-time setup (opt-in shared-memory limits of the tcgen05 and video_rows kernels); call with the device current
cudaError_t umma_conv_device_init();
cudaError_t video_rows_device_init();

// ---- planar-layout glue --------------------------------------------------------------------------
// fp32 channels-last (N,T,H,W,C) -> padded planar bf16 (plain, or parity-split when parity != 0); pads are NOT written.
void launch_pack_planar(const float* x, __nv_bfloat16* y, int64_t plane_stride, int64_t set_stride, UcGeom g, UcGeom g2, int C,
                        int parity, cudaStream_t s);
// padded planar bf16 (plain) -> fp32 channels-last rows (valid positions only)
void launch_unpack_planar(const __nv_bfloat16* x, int64_t plane_stride, UcGeom g, int C, float* y, int ld, cudaStream_t s);
// introspection: plain or parity-split planar buffer (+ optional low part) -> fp32 channels-last (N, T, Hf, Wf, C)
void launch_unpack_planar_any(const __nv_bfloat16* x, const __nv_bfloat16* xlo, int64_t plane_stride, int64_t set_stride, UcGeom g, int C, int sets,
                              int Hf, int Wf, float* y, cudaStream_t s);
// mean over `group` consecutive valid positions -> fp32 y[(row) * ld + c]; per_window != 0: one row per window (mean over T*H*W),
// else one row per (n,t) (mean over H*W).
void launch_planar_mean(const __nv_bfloat16* x, int64_t plane_stride, UcGeom g, int C, float* y, int ld, int per_window, cudaStream_t s);
// temporal difference in planar layout: d[n,t] = x[n,t+1] - x[n,t]  (geometry gd has T-1 frames)
void launch_planar_delta(const __nv_bfloat16* x, int64_t x_plane_stride, UcGeom g, __nv_bfloat16* d, int64_t d_plane_stride, UcGeom gd,
                         int C, cudaStream_t s);
// 3x3 / stride 2 / pad 1 max-pool over (H,W) in planar layout (plain -> plain); valid positions only
void launch_planar_maxpool(const __nv_bfloat16* x, int64_t x_plane_stride, UcGeom gi, __nv_bfloat16* y, int64_t y_plane_stride, UcGeom go,
                           int C, cudaStream_t s, const __nv_bfloat16* xlo = nullptr, __nv_bfloat16* ylo = nullptr);

// video (any dtype; NCDHW or NDHWC; uint8 scaled by 1/255) -> bf16 pixel rows xs (stem input) and xl = per-frame 3x3 conv 3->3
// with weights lapw [tap][ci][co] (artifact_detector.py:33-35,55-57).  Row layout: h-parity plane sets, geometry g (units of
// 2 pixels), pixel p of a row at element offset (p + 4) * 4, channels (r, g, b, 0).
// starts != nullptr (interleaved tracks, bulk-copy path only — check video_rows_bulk_ok): window n reads frames
// starts[n] .. starts[n]+T-1 of an n_frames-long track instead of frames n*T .. n*T+T-1.
// lapw_host: the same 81 weights on the host; the bulk-copy kernel takes them by value (constant-bank FFMA operands instead of 81
// shared-memory loads per 4 pixels).
void launch_video_rows(const void* video, int dtype, int layout, const float* lapw, const float* lapw_host, __nv_bfloat16* xs, __nv_bfloat16* xl,
                       int64_t set_stride, UcGeom g, int H, int W, cudaStream_t s, int num_sms, const int32_t* starts = nullptr, int n_frames = 0);
bool video_rows_bulk_ok(const void* video, int dtype, int layout, int W);

inline UcGeom make_geom_ex(int N, int T, int H, int W, int tpad, int oh, int hp_extra, int ow, int wp_extra) {
  UcGeom g;
  g.N = N; g.T = T; g.H = H; g.W = W;
  g.TS = T + tpad; g.ot = tpad;
  g.HP = H + oh + hp_extra; g.oh = oh;
  g.RW = W + ow + wp_extra; g.ow = ow;
  g.SL = g.HP * g.RW;
  g.P_total = ((int64_t)N * g.TS + tpad) * g.SL;
  uc_magic((uint32_t)g.SL, g.mSL, g.sSL);
  uc_magic((uint32_t)g.RW, g.mRW, g.sRW);
  uc_magic((uint32_t)g.TS, g.mTS, g.sTS);
  return g;
}
inline UcGeom make_geom(int N, int T, int H, int W) { return make_geom_ex(N, T, H, W, 1, 1, 0, 1, 0); }
// plain row-major rows (Linear layers): P == row
inline UcGeom make_geom_rows(int rows) { return make_geom_ex(1, 1, 1, rows, 0, 0, 0, 0, 0); }

}  // namespace lsd
