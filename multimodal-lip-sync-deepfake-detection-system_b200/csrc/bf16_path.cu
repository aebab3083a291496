// bf16 tensor-core path: weight packing for the tcgen05 flat shift-GEMM kernel (umma_conv.cu) and the forward
// orchestration that runs the 3-D residual stages, the artifact-detector convolutions and the high-frequency
// back end on it.  Host-side only.
#include "forward_common.h"
#include "tok_front.cuh"
#include "tok_fused.cuh"
#include "token_kernels.cuh"
#include "umma_conv.cuh"
#include "stem_ring.cuh"

#include <cuda_fp16.h>

#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>

using namespace lsd;
using namespace lsdfw;

// Environment knobs are read once per process (a getenv per knob per launch was ~0.2 ms of host time per forward); the A/B and
// trace switches that tests and experiments flip inside one process (LSD_TOK_FRONT / LSD_TOK_FUSED, *_TRACE, *_SKIP) stay live.
#define LSD_ENV(name) ([]() -> const char* { static const char* const v_ = getenv(name); return v_; }())

namespace {

uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);
  u += 0x7FFFu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

// Tap/band structure of a k_t x k_h x k_w convolution with stride (1, sh, sw) and "same" padding k/2 over the padded
// planar layout: taps that read the same parity plane set and the same temporal offset form one band.
// merge_kt: taps of all temporal offsets that read the same parity set share one band (small maps: the three temporal
// slabs of a tile are close together, so one region covers them and the stage carries up to 12 taps).
BGroup make_group(const ConvP& c, int sh, int sw, bool merge_kt = false) {
  BGroup g;
  g.Cin = c.Cin;
  for (int a = 0; a < c.kt; ++a)
    for (int b = 0; b < c.kh; ++b)
      for (int d = 0; d < c.kw; ++d) {
        BTap t;
        t.orig = (a * c.kh + b) * c.kw + d;
        t.dt = a - c.kt / 2;
        int hp = 0, wp = 0;
        const int oh = b - c.kh / 2, ow = d - c.kw / 2;
        if (sh == 2) { hp = oh & 1; t.dh = (oh - hp) / 2; } else t.dh = oh;
        if (sw == 2) { wp = ow & 1; t.dw = (ow - wp) / 2; } else t.dw = ow;
        const int set = hp * 2 + wp;
        BBand* band = nullptr;
        for (BBand& bb : g.bands)
          if (bb.set == set && (merge_kt || bb.taps[0].dt == t.dt) && (int)bb.taps.size() < UC_MAX_TAPS) band = &bb;
        if (!band) { g.bands.push_back(BBand{set, {}}); band = &g.bands.back(); }
        band->taps.push_back(t);
      }
  g.taps_total = c.kt * c.kh * c.kw;
  g.k16 = c.Cin / 16;
  return g;
}

// Toeplitz group (Cin = 3 convolutions with stride 2 in w, reading bf16 "pixel rows": 4 channels x 2 B per pixel, h-parity
// split, 2 pixels per 16-byte unit): a "tap" is one (kt, kh) pair, K runs over `kpix` consecutive pixels of the input row
// starting at pixel 2*wo + kw0 - pad_w (kw0 = -1: one leading zero-weight pixel keeps the start 16-byte aligned).
BGroup make_group_toeplitz(const ConvP& c, int kpix, int dw_units) {
  BGroup g;
  g.Cin = c.Cin;
  g.toeplitz = 1;
  g.k16 = kpix * 4 / 16;
  for (int a = 0; a < c.kt; ++a)
    for (int b = 0; b < c.kh; ++b) {
      BTap t;
      t.orig = a * c.kh + b;
      t.dt = a - c.kt / 2;
      const int oh = b - c.kh / 2;
      const int hp = oh & 1;
      t.dh = (oh - hp) / 2;
      t.dw = dw_units;
      BBand* band = nullptr;
      for (BBand& bb : g.bands)
        if (bb.set == hp && bb.taps[0].dt == t.dt) band = &bb;
      if (!band) { g.bands.push_back(BBand{hp, {}}); band = &g.bands.back(); }
      band->taps.push_back(t);
    }
  g.taps_total = c.kt * c.kh;
  return g;
}

struct Packer {
  lsd_handle* h;
  const std::vector<float>& f32;
  std::vector<uint16_t> w;
  std::vector<float> bias;
  int ds_sh = 2, ds_sw = 2;   // stride of the downsample conv fused by the next add(..., ds_key)
  // packed order: [Cout slice][k16 chunk][tap in band order][2 k-chunks][ntile][8]
  // part: 0 = bf16(W*scale) ("hi"), 1 = bf16(W*scale - hi) ("lo")
  void pack_group(BGroup& g, const ConvP& c, int ntile, int part = 0) {
    g.w_off = w.size();
    const int Cout = c.Cout;
    const float* W = &f32[c.w_off];
    const float* sc = c.has_scale ? &f32[c.scale_off] : nullptr;
    g.slice_stride = (size_t)(c.Cin / 16) * g.taps_total * ntile * 16;
    for (int sl = 0; sl < Cout / ntile; ++sl)
      for (int ch = 0; ch < c.Cin / 16; ++ch)
        for (const BBand& b : g.bands)
          for (const BTap& t : b.taps)
            for (int kc = 0; kc < 2; ++kc)
              for (int nn = 0; nn < ntile; ++nn)
                for (int e = 0; e < 8; ++e) {
                  const int ci = ch * 16 + kc * 8 + e, n = sl * ntile + nn;
                  const float v = W[((size_t)t.orig * c.Cin + ci) * Cout + n] * (sc ? sc[n] : 1.0f);
                  const uint16_t hi = f2bf(v);
                  if (part == 0) w.push_back(hi);
                  else { uint32_t u = (uint32_t)hi << 16; float hf; memcpy(&hf, &u, 4); w.push_back(f2bf(v - hf)); }
                }
  }
  // Toeplitz packing: K index k = c*16 + kc*8 + e  <->  pixel j = k/4 of the row window, channel k%4; kw = j - 1.
  // dup_lo: single-channel input stored as (hi, lo) bf16 pair in channels 0/1 -> both channels carry the channel-0 weight
  // halves: the weights are packed as two slices of Cout/2 columns (CTA pairs stage one half each)
  void add_toeplitz(const std::string& name, const std::string& key, int kpix, int dw_units, bool dup_lo = false, bool halves = false) {
    const ConvP& c = h->convs.at(key);
    BLayer L;
    L.Cout = c.Cout;
    L.ntile = c.Cout;
    L.halves = halves;
    L.groups.push_back(make_group_toeplitz(c, kpix, dw_units));
    BGroup& g = L.groups[0];
    g.w_off = w.size();
    const float* W = &f32[c.w_off];
    const float* sc = c.has_scale ? &f32[c.scale_off] : nullptr;
    const int nsl = halves ? 2 : 1, ncol = c.Cout / nsl;
    g.slice_stride = (size_t)g.k16 * g.taps_total * ncol * 16;
    for (int sl = 0; sl < nsl; ++sl)
    for (int ch = 0; ch < g.k16; ++ch)
      for (const BBand& b : g.bands)
        for (const BTap& t : b.taps)
          for (int kc = 0; kc < 2; ++kc)
            for (int n = sl * ncol; n < (sl + 1) * ncol; ++n)
              for (int e = 0; e < 8; ++e) {
                const int k = ch * 16 + kc * 8 + e, j = k / 4, kw = j - 1;
                int ci = k % 4;
                const bool lo_part = dup_lo && ci == 2;     // channel 2 = x_hi again, multiplied by the low part of W
                if (dup_lo) ci = ci < 3 ? 0 : 99;
                float v = 0.f;
                if (ci < c.Cin && kw >= 0 && kw < c.kw) v = W[((size_t)(t.orig * c.kw + kw) * c.Cin + ci) * c.Cout + n] * (sc ? sc[n] : 1.0f);
                const uint16_t hi = f2bf(v);
                if (!lo_part) w.push_back(hi);
                else { uint32_t u = (uint32_t)hi << 16; float hf; memcpy(&hf, &u, 4); w.push_back(f2bf(v - hf)); }
              }
    L.bias_off = bias.size();
    for (int i = 0; i < c.Cout; ++i) bias.push_back(f32[c.shift_off + i]);
    while (w.size() % 64) w.push_back(0);
    h->blayers[name] = L;
  }
  // split: every K group is issued three times (hi*hi, lo*hi, hi*lo), see add_split
  void add(const std::string& name, const std::string& key, int sh, int sw, const std::string& ds_key = "", int ntile = 0, bool split = false,
           bool merge_kt = false, bool halves = false) {
    const ConvP& c = h->convs.at(key);
    BLayer L;
    L.Cout = c.Cout;
    L.ntile = ntile > 0 ? ntile : c.Cout;
    L.halves = halves;   // (single-group layers only)
    L.groups.push_back(make_group(c, sh, sw, merge_kt));
    pack_group(L.groups[0], c, halves ? L.ntile / 2 : L.ntile);
    if (split) {
      BGroup g1 = L.groups[0]; g1.src = 2;
      BGroup g2 = make_group(c, sh, sw, merge_kt);
      pack_group(g2, c, L.ntile, 1);
      L.groups.push_back(g1);
      L.groups.push_back(g2);
    }
    L.bias_off = bias.size();
    for (int i = 0; i < c.Cout; ++i) bias.push_back(f32[c.shift_off + i]);
    if (!ds_key.empty()) {
      const ConvP& d = h->convs.at(ds_key);
      const int sh_ds = ds_sh, sw_ds = ds_sw;
      BGroup gd = make_group(d, sh_ds, sw_ds);  // 1x1 strided conv reads parity set (0,0) with zero shift
      gd.src = 1;
      pack_group(gd, d, L.ntile);
      L.groups.push_back(gd);
      if (split) {
        BGroup g1 = gd; g1.src = 3;
        BGroup g2 = make_group(d, sh_ds, sw_ds); g2.src = 1;
        pack_group(g2, d, L.ntile, 1);
        L.groups.push_back(g1);
        L.groups.push_back(g2);
      }
      for (int i = 0; i < c.Cout; ++i) bias[L.bias_off + i] += f32[d.shift_off + i];
    }
    while (w.size() % 64) w.push_back(0);
    h->blayers[name] = L;
  }
  // The same 3x3x3 convolution (+ fused 1x1 downsample) for the folded small-map route (UcFoldSlice in umma_conv.cuh): the taps
  // are packed in (kh, kw, kt) order, so the three temporal taps of one spatial tap — one band of a folded conv, A from the plane
  // set of one input position — are one contiguous weight piece per K chunk.  Same bf16 values as the padded route's packing.
  void add_fold(const std::string& name, const std::string& key, const std::string& ds_key, int ntile) {
    const ConvP& c = h->convs.at(key);
    if (c.kt != 3 || c.kh != 3 || c.kw != 3 || c.Cout % ntile) return;
    BLayer L;
    L.Cout = c.Cout;
    L.ntile = ntile;
    BGroup g;
    g.Cin = c.Cin;
    g.taps_total = 27;
    g.k16 = c.Cin / 16;
    for (int b = 0; b < 3; ++b)
      for (int d = 0; d < 3; ++d) {
        BBand band{b * 3 + d, {}};
        for (int a = 0; a < 3; ++a) band.taps.push_back(BTap{(a * 3 + b) * 3 + d, a - 1, b - 1, d - 1});
        g.bands.push_back(band);
      }
    pack_group(g, c, ntile);
    L.groups.push_back(g);
    L.bias_off = bias.size();
    for (int i = 0; i < c.Cout; ++i) bias.push_back(f32[c.shift_off + i]);
    if (!ds_key.empty()) {
      const ConvP& d = h->convs.at(ds_key);
      BGroup gd = make_group(d, 1, 1);
      gd.src = 1;
      pack_group(gd, d, ntile);
      L.groups.push_back(gd);
      for (int i = 0; i < c.Cout; ++i) bias[L.bias_off + i] += f32[d.shift_off + i];
    }
    while (w.size() % 64) w.push_back(0);
    h->blayers[name] = L;
  }
  // Split-bf16 ("bf16x3") layer for the token path: y = Ahi*Whi + Alo*Whi + Ahi*Wlo accumulated in one TMEM tile
  // (three K groups), which keeps ~16 mantissa bits of both operands; the dropped Alo*Wlo term is ~2^-16 relative.
  void add_split(const std::string& name, const std::string& key, int ntile) {
    const ConvP& c = h->convs.at(key);
    BLayer L;
    L.Cout = c.Cout;
    L.ntile = ntile;
    BGroup g0 = make_group(c, 1, 1);
    pack_group(g0, c, ntile, 0);
    BGroup g1 = g0; g1.src = 2;                 // low part of the activations x the same high weights
    BGroup g2 = make_group(c, 1, 1);
    pack_group(g2, c, ntile, 1);                // high part of the activations x low weights
    L.groups = {g0, g1, g2};
    L.bias_off = bias.size();
    for (int i = 0; i < c.Cout; ++i) bias.push_back(f32[c.shift_off + i]);
    while (w.size() % 64) w.push_back(0);
    h->blayers[name] = L;
  }
};

// ---- planar activation buffers ----------------------------------------------------------------
struct PBuf {
  size_t off = 0;          // byte offset into the workspace
  int C = 0, sets = 1;
  int kind = PK_PLAIN;     // layout (PlanarKind) and full-resolution map extent: what lsd_planar_stage_read accepts
  int map_h = 0, map_w = 0;
  UcGeom g;                // geometry of each plane set
  int64_t plane_stride = 0, set_stride = 0, origin = 0;  // elements
  size_t bytes() const { return (size_t)sets * set_stride * 2; }
};

constexpr int TILE_MAX = 1024;  // largest MT*128

PBuf make_pbuf(int C, int sets, UcGeom g) {
  PBuf b;
  b.C = C; b.sets = sets; b.g = g;
  const int64_t gf = ((int64_t)g.SL + 3 * g.RW + 16 + 7) / 8 * 8;
  const int64_t gb = gf + TILE_MAX;
  const int64_t plane_pos = (gf + g.P_total + gb + 7) / 8 * 8;
  b.origin = gf * 8;
  b.plane_stride = plane_pos * 8;
  b.set_stride = b.plane_stride * (C / 8);
  return b;
}

// Folded route (UcFoldSlice in umma_conv.cuh) for the residual stage whose output map is H x W: on small maps the padded layout
// executes 49 positions per 36 (6x6) or 16 per 9 (3x3) and multiplies every tap, including those that only read padding.  Chosen
// from the geometry alone (never from the batch); LSD_FOLD=0 keeps the padded route everywhere (reference for A/B runs).
bool fold_route(int H, int W) {
  static const bool off = LSD_ENV("LSD_FOLD") && atoi(LSD_ENV("LSD_FOLD")) == 0;
  return !off && H * W <= 36;
}

struct BPlan {
  Shapes s;
  bool fold3 = false, fold4 = false;      // layer3 / layer4 on the folded route
  Plan f32;                               // fp32 buffers (stage registry + bump allocator)
  std::map<std::string, PBuf> pb;
  size_t planar_begin = 0, planar_end = 0;
  UcGeom gt, g33, gta;                    // token geometries: T tokens (+3 pad), T+1 tokens (rows), audio tokens (rows)
  // kind PK_PLAIN: the map is the plane geometry itself; the other kinds name the map extent (mh, mw) they hold
  void addp(const char* name, int C, int sets, UcGeom g, int kind = PK_PLAIN, int mh = 0, int mw = 0) {
    PBuf b = make_pbuf(C, sets, g);
    b.kind = kind;
    b.map_h = kind == PK_PLAIN ? g.H : mh;
    b.map_w = kind == PK_PLAIN ? g.W : mw;
    f32.cursor = (f32.cursor + 255) & ~size_t(255);
    b.off = f32.cursor;
    f32.cursor += b.bytes();
    pb[name] = b;
  }
};

// video = false: the audio side of the shared-visual forward (see VarTail), which runs the audio encoder and the fused token
// kernels only: no video input, no visual-encoder, visual-token, aux or launch-by-launch token-path buffers
void build_plan(const Shapes& s, BPlan& P, bool video = true) {
  P.s = s;
  Plan& p = P.f32;
  const int64_t B = s.B, T = s.T, TA = s.A4;
  if (video) p.add("vid", B * T * s.H * s.W * 3);     // only used by the uint8-track window builder (lsd_score_windows)
  p.add("aud", B * s.F * s.Ta);
  if (video) p.add("v_feat", B * T * 256);
  p.add("a_feat", B * TA * 256);
  if (video) {
  p.add("v_emb", B * T * 256);
  p.add("a_emb", B * TA * 256);
  p.add("a_int", B * T * 256);
  p.add("proj_v", B * T * 768);
  p.add("proj_a", B * T * 768);
  p.add("vcomb", B * T * 1024);            // [v_emb | in-projection of the visual tokens] per token (fused token path)
  }
  p.add("acomb", B * T * 1024);            // [interpolated a_emb | in-projection of the interpolated audio tokens]
  p.add("a_fint", B * T * 256);            // audio features interpolated to T tokens
  p.add("gate_in", B * T * 512);
  if (video) p.add("gate_h", B * T * 256);
  p.add("fused", B * T * 256);
  p.add("tok", B * (T + 1) * 256);
  if (video) {
  p.add("tok_qkv", B * (T + 1) * 768);
  p.add("comb", B * 448);
  }
  // planar bf16 buffers
  P.planar_begin = (p.cursor + 255) & ~size_t(255);
  const int Bn = s.B, Tn = s.T;
  const UcGeom g1 = make_geom(Bn, Tn, s.H1, s.W1), g2 = make_geom(Bn, Tn, s.H2, s.W2), g3 = make_geom(Bn, Tn, s.H3, s.W3),
               g4 = make_geom(Bn, Tn, s.H4, s.W4), gd = make_geom(Bn, s.Td, s.H4, s.W4), gh = make_geom(Bn, Tn, s.Hg, s.Wg);
  // bf16 pixel rows of the video and of its per-frame 3->3 "laplacian" conv (h-parity split; 16-byte unit = 2 pixels x 4 ch)
  // (row = 2 zero units + W/2 data units: the 2 leading units of the NEXT row are this row's right padding — the 7-tap window of the
  //  last output reaches one unit past the data — so the row pitch is W/2 + 2, not W/2 + 4: 4 % fewer positions for the stem and hf0)
  const UcGeom gs = make_geom_ex(Bn, Tn, s.Hs, s.Ws, 1, 2, 0, 0, 2);
  if (video) {
  P.addp("xs", 8, 2, gs, PK_ROWS, s.H, s.W);
  P.addp("xl", 8, 2, gs, PK_ROWS, s.H, s.W);
  P.addp("s_out", 64, 1, gs);    // stem conv output (stem geometry), before the max-pool
  P.addp("x1", 64, 1, g1);
  P.addp("l1a", 64, 1, g1);
  P.addp("y1", 64, 4, g2, PK_PARITY_HW, s.H1, s.W1);   // parity-split: four half-resolution plane sets
  P.addp("l2a", 128, 1, g2);
  // folded route (small maps): y2 / l3a / y3 / l4a hold one plane set per map position in the row geometry gr
  P.fold3 = fold_route(s.H3, s.W3);
  P.fold4 = fold_route(s.H4, s.W4);
  const UcGeom gr = make_geom_ex(Bn, Tn, 1, 1, 1, 0, 0, 0, 0);
  if (P.fold3) P.addp("y2", 128, s.H2 * s.W2, gr, PK_FOLD, s.H2, s.W2); else P.addp("y2", 128, 4, g3, PK_PARITY_HW, s.H2, s.W2);
  if (P.fold3) P.addp("l3a", 256, s.H3 * s.W3, gr, PK_FOLD, s.H3, s.W3); else P.addp("l3a", 256, 1, g3);
  if (P.fold4) P.addp("y3", 256, s.H3 * s.W3, gr, PK_FOLD, s.H3, s.W3); else P.addp("y3", 256, 4, g4, PK_PARITY_HW, s.H3, s.W3);
  if (P.fold4) P.addp("l4a", 256, s.H4 * s.W4, gr, PK_FOLD, s.H4, s.W4); else P.addp("l4a", 256, 1, g4);
  P.addp("y4", 256, 1, g4);
  P.addp("art_a", 128, 1, g4);
  P.addp("art_b", 64, 1, g4);
  P.addp("delta", 256, 1, gd);
  P.addp("artd_a", 128, 1, gd);
  P.addp("artd_b", 64, 1, gd);
  P.addp("hf_f", 32, 4, gh, PK_PARITY_HW, s.Hh, s.Wh);
  P.addp("hf_b", 64, 1, gh);
  }
  // audio encoder: 2-D geometries (one slab per window, no temporal padding)
  const UcGeom as = make_geom_ex(Bn, 1, s.Fs, s.As, 0, 2, 0, 0, 4);
  auto g2d = [&](int H, int W) { return make_geom_ex(Bn, 1, H, W, 0, 1, 0, 1, 0); };
  P.addp("xa", 8, 2, as, PK_ROWS, s.F, s.Ta);
  for (const char* sfx : {"", "_lo"}) {      // audio activations are (hi, lo) bf16 pairs (split-bf16 convolutions)
    auto nm = [&](const char* n) { return std::string(n) + sfx; };
    P.addp(nm("sa_out").c_str(), 64, 1, as);
    P.addp(nm("a1").c_str(), 64, 1, g2d(s.F1, s.A1));
    P.addp(nm("a1a").c_str(), 64, 1, g2d(s.F1, s.A1));
    P.addp(nm("ya1").c_str(), 64, 4, g2d(s.F2, s.A2), PK_PARITY_HW, s.F1, s.A1);
    P.addp(nm("a2a").c_str(), 128, 1, g2d(s.F2, s.A2));
    P.addp(nm("ya2").c_str(), 128, 4, g2d(s.F3, s.A3), PK_PARITY_H, s.F2, s.A2);   // h-parity only (stride (2,1)): sets 0 and 2 are used
    P.addp(nm("a3a").c_str(), 256, 1, g2d(s.F3, s.A3));
    P.addp(nm("ya3").c_str(), 256, 4, g2d(s.F4, s.A4), PK_PARITY_H, s.F3, s.A3);
    P.addp(nm("a4a").c_str(), 256, 1, g2d(s.F4, s.A4));
    P.addp(nm("ya4").c_str(), 256, 1, g2d(s.F4, s.A4));
  }
  // token path
  P.gt = make_geom_ex(Bn, 1, 1, Tn, 0, 0, 0, 3, 0);   // 3 zero positions before every window (conv1d k<=7)
  P.g33 = make_geom_rows(Bn * (Tn + 1));
  P.gta = make_geom_rows(Bn * (int)TA);
  // every token-path GEMM operand exists as a (hi, lo) bf16 pair ("<name>" / "<name>_lo")
  for (const char* sfx : {"", "_lo"}) {
    auto nm = [&](const char* n) { return std::string(n) + sfx; };
    P.addp(nm("afeat_p").c_str(), 256, 1, P.gta);
    if (!video) { P.addp(nm("afint_p").c_str(), 256, 1, P.gt); continue; }
    for (const char* n : {"vfeat_p", "vemb_p", "aint_p", "afint_p", "att1_p", "att2_p", "blend_p", "fused_p"}) P.addp(nm(n).c_str(), 256, 1, P.gt);
    P.addp(nm("gatein_p").c_str(), 512, 1, P.gt);
    P.addp(nm("mscat_p").c_str(), 768, 1, P.gt);
    P.addp(nm("tokln_p").c_str(), 256, 1, P.g33);
    P.addp(nm("tokatt_p").c_str(), 256, 1, P.g33);
    P.addp(nm("tokff_p").c_str(), 1024, 1, P.g33);
  }
  P.planar_end = p.cursor;
}

struct BCtx {
  lsd_handle* h;
  char* ws;
  const BPlan* P;
  cudaStream_t st;
  int max_ctas = 0;        // > 0: persistent grids of this context are limited (side stream shares the GPU with the main one)
  __nv_bfloat16* base(const PBuf& b) const { return reinterpret_cast<__nv_bfloat16*>(ws + b.off); }
  __nv_bfloat16* org(const PBuf& b) const { return base(b) + b.origin; }
  float* f(const char* name) const { return reinterpret_cast<float*>(ws + P->f32.find(name)); }
  const float* W(const char* key) const { return h->warena + h->vecs.at(key); }
};

struct UArgs {
  const PBuf* in = nullptr;       // main input (planar, or pixel rows for Toeplitz layers)
  const PBuf* in_ds = nullptr;    // input of the fused strided 1x1 downsample group
  const PBuf* in_lo = nullptr;    // low part of the main input (split-bf16 layers)
  const PBuf* in_ds_lo = nullptr; // low part of the downsample input
  const PBuf* res_lo = nullptr;   // low part of the residual
  const PBuf* yp_lo = nullptr;    // low part of the planar destination
  UcGeom og;                      // output geometry (== flat geometry of every input band)
  int act = ACT_NONE;
  const PBuf* yp = nullptr;       // planar bf16 destination (plain when sets == 1, parity-split when 4)
  int y_plane_off = 0;            // first destination plane (concatenation along channels)
  int y_mode = -1;                // -1: derive from yp->sets
  const PBuf* res = nullptr;      // bf16 residual (plain, output geometry)
  float* y32 = nullptr;           // fp32 row destination
  int y32_ld = 0, y32_outer_stride = -1, y32_row_off = 0;
  const float* res32 = nullptr;   // fp32 row residual (compact rows)
  int res32_ld = 0;
};

// Stage program of a launch: expanded on the host by `build`, cached in device memory under a hash of the complete parameter block
// (pointers, strides, geometry, tile shape, fold slices), so steady-state forwards only look it up.  Sets p.prog.
// salt: what else the program depends on (folded convs: input map extents and set strides, which the parameter block does not hold)
int stage_program(const BCtx& c, const std::string& name, UmmaConvP& p, const std::function<void(std::vector<UcStageDesc>&)>& build,
                  std::initializer_list<uint64_t> salt = {}) {
  uint64_t hkey = 1469598103934665603ull;
  for (uint64_t v : salt) { hkey ^= v; hkey *= 1099511628211ull; hkey ^= hkey >> 29; }
  static_assert(sizeof(UmmaConvP) % 8 == 0, "UmmaConvP is hashed in 8-byte words");
  const uint64_t* pw = reinterpret_cast<const uint64_t*>(&p);   // (p was memset to 0 first: padding bytes are deterministic)
  for (size_t i = 0; i < sizeof(p) / 8; ++i) { hkey ^= pw[i]; hkey *= 1099511628211ull; hkey ^= hkey >> 29; }
  auto it = c.h->prog_cache.find(hkey);
  if (it == c.h->prog_cache.end()) {
    std::vector<UcStageDesc> host;
    build(host);
    const size_t bytes = host.size() * sizeof(UcStageDesc);
    if (!c.h->prog_arena) {
      c.h->prog_cap = 64u << 20;   // (a folded conv's slice programs are ~0.3 MB per shape and workspace)
      if (cudaMalloc(&c.h->prog_arena, c.h->prog_cap) != cudaSuccess) return lsd_fail(c.h, LSD_ERR_CUDA, "stage-program arena allocation failed");
      c.h->prog_cursor = 0;
    }
    if (c.h->prog_cursor + bytes > c.h->prog_cap) {   // arena full (many shapes / workspaces seen): start over once nothing is in flight
      cudaDeviceSynchronize();
      c.h->prog_cache.clear();
      c.h->prog_cursor = 0;
      ++c.h->generation;   // captured CUDA graphs hold addresses of the old programs
    }
    char* dst = c.h->prog_arena + c.h->prog_cursor;
    // Cache miss only (first forward of a shape): a blocking copy, so the program is visible to every stream that later
    // launches this layer (the cache is shared by the main, side, tail and helper streams).
    cudaError_t e = cudaMemcpy(dst, host.data(), bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return lsd_fail(c.h, LSD_ERR_CUDA, "%s: stage program upload: %s", name.c_str(), cudaGetErrorString(e));
    c.h->prog_cursor += (bytes + 255) & ~size_t(255);
    it = c.h->prog_cache.emplace(hkey, dst).first;
  }
  p.prog = reinterpret_cast<const UcStageDesc*>(it->second);
  return 0;
}

// One launch of the tcgen05 kernel for layer `name`.
int run_umma(const BCtx& c, const std::string& name, const UArgs& a) {
  const BLayer& L = c.h->blayers.at(name);
  const UcGeom& og = a.og;
  if (og.P_total >= ((int64_t)1 << 31) - 1024) return lsd_fail(c.h, LSD_ERR_SHAPE, "%s: more than 2^31 padded positions in one launch (reduce the batch)", name.c_str());
  UmmaConvP p;
  memset(&p, 0, sizeof(p));
  p.w = reinterpret_cast<const __nv_bfloat16*>(c.h->barena);
  p.bias = c.h->bbias + L.bias_off;
  p.Cout = L.ntile;
  const int slices = L.Cout / L.ntile;
  p.act = a.act;
  p.g = og;
  p.cta2 = L.halves ? 1 : 0;
  if (a.yp) {
    p.y_mode = a.y_mode >= 0 ? a.y_mode : (a.yp->sets == 4 ? UC_Y_PARITY : UC_Y_PLAIN);
    p.y = c.org(*a.yp) + (int64_t)a.y_plane_off * a.yp->plane_stride;
    p.y_plane_stride = a.yp->plane_stride; p.y_set_stride = a.yp->set_stride;
    p.g2 = a.yp->g;
    p.ymap_W = og.W;
    if (a.yp_lo) p.ylo = c.org(*a.yp_lo) + (int64_t)a.y_plane_off * a.yp_lo->plane_stride;
  }
  if (a.y32) {
    p.y32 = a.y32; p.y32_ld = a.y32_ld;
    p.y32_outer_stride = a.y32_outer_stride >= 0 ? a.y32_outer_stride : og.W;
    p.y32_row_off = a.y32_row_off;
  }
  if (a.res) { p.res = c.org(*a.res); p.res_plane_stride = a.res->plane_stride; }
  if (a.res_lo) p.res_lo = c.org(*a.res_lo);
  if (a.res32) { p.res32 = a.res32; p.res32_ld = a.res32_ld; }
  // Tile shape.  The kernel is bound by shared-memory bandwidth (operand reads of the MMAs + the fills of the ring), so
  // the fills per MMA are minimised: wide layers (>= 128 columns) give all 512 TMEM columns to one tile (more M-tiles per
  // weight stage; their K loop is so long that the un-overlapped epilogue is a few %), narrow layers keep two
  // accumulator buffers so that the epilogue overlaps the next tile.  MT shrinks while the tiles cannot fill the SMs.
  // (32-column layers — the hf front convolution — take 8 M-tiles: their stages carry one MMA per M-tile, so an issuing warp's
  // per-stage cost, ~300 cycles of barrier / descriptor bookkeeping, is what bounds them; two M-tiles per issuer halve it)
  const int mt_cap = L.ntile <= 32 ? 8 : 4;
  const int mt2 = std::max(1, std::min(mt_cap, 256 / L.ntile));   // M-tiles per tile with two accumulator buffers
  p.MT = std::max(1, std::min(mt_cap, 512 / L.ntile));             // ... with one
  // (the CTAs this launch may use: side-stream launches are capped, and a cap of 74 with 265 one-M-tile tiles meant four waves of
  // single-issuer tiles where two waves of two-M-tile tiles do — the artifact convolutions on the 3x3 maps)
  const int cta_budget = (c.max_ctas > 0 && c.max_ctas < c.h->num_sms) ? c.max_ctas : c.h->num_sms;
  while (p.MT > 1 && ((og.P_total + p.MT * 128 - 1) / (p.MT * 128)) * slices < cta_budget) p.MT /= 2;
  p.nbuf = (p.MT <= mt2 && 2 * p.MT * L.ntile <= 512) ? 2 : 1;  // single buffering only when it buys a larger tile
  if (const char* e = LSD_ENV("LSD_UMMA_NBUF")) {               // tuning knob
    const int v = atoi(e);
    if (v == 1) p.nbuf = 1;
    if (v == 2 && 2 * L.ntile <= 512) { p.nbuf = 2; p.MT = std::min(p.MT, mt2); }
  }
  // One issue-loop iteration (one tap: descriptor arithmetic + R2UR moves + the MMAs) costs an issuing warp 150-260 cycles,
  // more than the tensor time of the MMAs it carries for narrow tiles, so the M-tiles of a tap are spread over as many
  // issuing warps as there are M-tiles.
  p.issuers = std::min(p.MT, 4);   // (measured: one issuer for MT = 4 is 6-15 % slower than two on every layer)
  if (const char* e = LSD_ENV("LSD_UMMA_ISSUERS")) { const int v = atoi(e); if (v >= 1 && v <= 4 && v <= p.MT && p.MT % v == 0 && p.MT / v <= 4) p.issuers = v; }   // tuning knob
  uint32_t cols = 32;
  while ((int)cols < p.nbuf * p.MT * L.ntile) cols *= 2;
  p.tmem_cols = cols;
  const int S = p.MT * 128;
  int nb = 0, max_a = 0, max_taps = 0, min_k16 = 1 << 30;
  bool any_toeplitz = false;
  p.ngroups = (int)L.groups.size();
  for (int gi = 0; gi < p.ngroups; ++gi) {
    const BGroup& G = L.groups[gi];
    const PBuf* srcp = G.src == 0 ? a.in : (G.src == 1 ? a.in_ds : (G.src == 2 ? a.in_lo : a.in_ds_lo));
    if (!srcp) return lsd_fail(c.h, LSD_ERR_ARG, "%s: missing input for group %d", name.c_str(), gi);
    const PBuf& src = *srcp;
    UcGroup& ug = p.groups[gi];
    ug.band_begin = nb;
    ug.k16 = G.k16;
    ug.taps_total = G.taps_total;
    ug.w_off = (int64_t)G.w_off;
    ug.slice_stride = (int64_t)G.slice_stride;
    int tap_begin = 0;
    int wkb = 40;                                                                        // keep a weight stage <= ~40 KB
    if (const char* e = LSD_ENV("LSD_UMMA_WKB")) wkb = std::max(8, atoi(e));               // tuning knob
    const int tmax = std::max(1, std::min(UC_MAX_TAPS, (wkb * 1024) / (L.ntile * 32)));
    for (const BBand& b : G.bands) {
      const int nt = (int)b.taps.size();
      const int pieces = (nt + tmax - 1) / tmax, per = (nt + pieces - 1) / pieces;
      for (int t0 = 0; t0 < nt; t0 += per) {
        const int t1 = std::min(nt, t0 + per);
        if (nb >= UC_MAX_BANDS) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: too many bands", name.c_str());
        UcBand& ub = p.bands[nb++];
        ub.base = c.org(src) + (int64_t)b.set * src.set_stride;
        ub.plane_stride = src.plane_stride;
        ub.toeplitz = G.toeplitz;
        ub.chunk_stride = G.toeplitz ? 16 : 2 * src.plane_stride;
        int mn = INT32_MAX, mx = INT32_MIN;
        for (int j = t0; j < t1; ++j) {
          const BTap& t = b.taps[j];
          const int sft = t.dt * og.SL + t.dh * og.RW + t.dw;
          mn = std::min(mn, sft); mx = std::max(mx, sft);
        }
        ub.start = mn;
        ub.len_extra = mx - mn;
        ub.ntaps = t1 - t0;
        ub.tap_begin = tap_begin;
        for (int j = t0; j < t1; ++j) ub.rel[j - t0] = b.taps[j].dt * og.SL + b.taps[j].dh * og.RW + b.taps[j].dw - mn;
        tap_begin += ub.ntaps;
        max_a = std::max(max_a, G.toeplitz ? (S + ub.len_extra + 1 + 2 * (G.k16 - 1)) * 16 : 2 * (S + ub.len_extra) * 16);
        max_taps = std::max(max_taps, ub.ntaps);
        min_k16 = std::min(min_k16, G.k16);
        any_toeplitz = any_toeplitz || G.toeplitz;
        // the band must stay inside the guard zones of the source buffer
        if (-(int64_t)ub.start * 8 > src.origin || (int64_t)mx * 8 > src.origin)
          return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: guard zone too small", name.c_str());
      }
    }
    ug.band_end = nb;
  }
  p.nbands = nb;
  // K chunks per stage: Toeplitz layers share one row region for all chunks; small planar stages are packed up to ~24 KB
  const int w_chunk = max_taps * (L.halves ? L.ntile / 2 : L.ntile) * 32;   // (CTA pairs stage half of the columns per CTA)
  if (any_toeplitz) p.kpack = min_k16;
  else {
    // A stage costs its issuing warp ~300-450 cycles of barrier / descriptor bookkeeping whatever it carries: with 24 KB stages the
    // one-tap token GEMMs issued 4 MMAs per stage, ~145 cycles per MMA against 48 of tensor time (measured per step at B=64 with
    // 24 / 36 / 48 / 64 KB stages everywhere: 3.140 / 3.101 / 3.107 / 3.068 ms).  Only single-band layers (Linear) get the large
    // stages: with several bands the K accumulation order is (chunk block, band, chunk, tap), i.e. it depends on kpack, kpack
    // depends on the tile size and the tile size on the batch — logits must not depend on the batch composition bit for bit.
    bool single_band = true;
    for (int gi = 0; gi < p.ngroups; ++gi) single_band = single_band && (p.groups[gi].band_end - p.groups[gi].band_begin) == 1;
    int stage_kb = single_band ? 64 : 24;
    if (const char* e = LSD_ENV("LSD_UMMA_STAGE_KB")) stage_kb = std::max(8, atoi(e));   // tuning knob
    p.kpack = std::max(1, std::min(std::min(8, min_k16), (stage_kb * 1024) / (max_a + w_chunk)));
  }
  p.a_stage_bytes = ((uint32_t)(any_toeplitz ? max_a : max_a * p.kpack) + 127u) & ~127u;
  p.w_stage_bytes = (uint32_t)(w_chunk * p.kpack);
  const uint32_t stage = p.a_stage_bytes + p.w_stage_bytes;
  // stage program (one 64-byte descriptor per ring stage of a tile) lives behind the ring in shared memory
  p.nst_tile = 0;
  for (int gi = 0; gi < p.ngroups; ++gi)
    p.nst_tile += ((p.groups[gi].k16 + p.kpack - 1) / p.kpack) * (p.groups[gi].band_end - p.groups[gi].band_begin);
  const uint32_t prog_bytes = (uint32_t)p.nst_tile * (uint32_t)umma_conv_stage_desc_bytes();
  uint32_t budget = 211u * 1024u;   // one persistent CTA per SM owns the whole shared memory
  const uint32_t extra_bytes = (uint32_t)umma_conv_extra_smem_bytes(p);   // bias operand tiles of the lean epilogue
  budget -= extra_bytes;
  if (prog_bytes + 2 * stage > budget) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: stage program of %u bytes does not fit", name.c_str(), prog_bytes);
  int stages = (int)((budget - prog_bytes) / stage);
  stages = std::max(2, std::min(stages, 8));
  if ((size_t)stages * stage + prog_bytes + extra_bytes + 1024 > 223u * 1024u) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: stage of %u bytes does not fit", name.c_str(), stage);
  p.stages = stages;
  double kflop = 0;
  for (const BGroup& G : L.groups) kflop += (double)G.taps_total * G.Cin;
  if (L.groups[0].toeplitz) { const ConvP& cp = c.h->convs.at(name); kflop = (double)cp.kt * cp.kh * cp.kw * cp.Cin; }  // algorithmic K, not the padded one
  if (const char* e = getenv("LSD_UMMA_SKIP")) p.skip = atoi(e);
  if (const char* why = umma_conv_config_error(p)) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: %s", name.c_str(), why);
  if (int rc = stage_program(c, name, p, [&](std::vector<UcStageDesc>& v) { v.resize((size_t)p.nst_tile); umma_conv_build_program(p, v.data()); }))
    return rc;
  if (const char* e = getenv("LSD_UMMA_TRACE")) {
    // debug: per-launch phase timestamps of CTA (0,0); prints after a sync (never enabled in timed runs)
    static long long* dbuf = nullptr;
    if (!dbuf) cudaMalloc(&dbuf, 512);
    cudaMemsetAsync(dbuf, 0, 512, c.st);
    p.dbg = dbuf;
    launch_umma_conv(p, slices, c.st, c.h->num_sms, c.max_ctas);
    long long hv[64];
    cudaMemcpyAsync(hv, dbuf, 512, cudaMemcpyDeviceToHost, c.st);
    cudaStreamSynchronize(c.st);
    if (atoi(e) > 0)
      fprintf(stderr, "[umma] %-34s MT=%d N=%d slices=%d stages=%d kpack=%d tiles=%lld | prologue %lld, first-data %lld, mma-issued %lld, acc-done %lld, epi-done %lld, total %lld cycles\n",
              name.c_str(), p.MT, p.Cout, slices, p.stages, p.kpack, hv[7], hv[1] - hv[0], hv[2] - hv[0], hv[3] - hv[0], hv[4] - hv[0], hv[5] - hv[0], hv[6] - hv[0]);
    if (atoi(e) > 1) {
      fprintf(stderr, "        full-wait done at:");
      for (int i = 0; i < 24 && hv[8 + i]; ++i) fprintf(stderr, " %lld", hv[8 + i] - hv[0]);
      fprintf(stderr, "\n        producer issue at:");
      for (int i = 0; i < 24 && hv[32 + i]; ++i) fprintf(stderr, " %lld", hv[32 + i] - hv[0]);
      fprintf(stderr, "\n        copies issued at: ");
      for (int i = 0; i < 8 && hv[56 + i]; ++i) fprintf(stderr, " %lld", hv[56 + i] - hv[0]);
      fprintf(stderr, "\n");
    }
    return 0;
  }
  // profile classes: 2 = 3-D conv visual encoder (stem + residual stages, 86 % of the FLOPs, runs alone on the GPU),
  //                  3 = every other tcgen05 launch (audio encoder, token GEMMs, artifact branch on the side stream)
  c.h->prof.begin(c.st, 2.0 * (double)og.N * og.T * og.H * og.W * L.Cout * kflop, name.rfind("visual_encoder.", 0) == 0 ? 2 : 3);
  launch_umma_conv(p, slices, c.st, c.h->num_sms, c.max_ctas);
  c.h->prof.end(c.st);
  return 0;
}

// Step table of the temporal-ring stem (stem_ring.cu) for geometry g: (column chunk, t) outputs numbered column-major, cut into
// equal contiguous ranges, one per accumulator slot; cached per (batch, frames, geometry, CTA budget).
int ring_table(const BCtx& c, const UcGeom& g, const lsd_handle::RingTab** out) {
  lsd_handle* h = c.h;
  const int T = g.T, CH = (g.SL + 127) / 128;
  const int64_t G = (int64_t)g.N * CH * T;
  const int budget = (c.max_ctas > 0 && c.max_ctas < h->num_sms) ? c.max_ctas : h->num_sms;
  uint64_t key = 1469598103934665603ull;
  for (uint64_t v : {(uint64_t)g.N, (uint64_t)T, (uint64_t)g.SL, (uint64_t)g.TS, (uint64_t)g.ot, (uint64_t)budget}) { key ^= v; key *= 1099511628211ull; key ^= key >> 29; }
  auto it = h->ring_tabs.find(key);
  if (it == h->ring_tabs.end()) {
    int grid = budget;
    int64_t Lr = (G + 2 * (int64_t)grid - 1) / (2 * (int64_t)grid);
    if (Lr < 8) { Lr = 8; grid = (int)((G + 2 * Lr - 1) / (2 * Lr)); }
    if (grid < 1) grid = 1;
    std::vector<std::vector<SrStep>> lists((size_t)2 * grid);
    size_t nsteps = 0;
    // steps of outputs [ta, tb) of column `col` (input slabs max(ta-1, 0) .. tb; the slab completed by a step is stored when it is in range)
    auto add_range = [&](int sg, int64_t col, int ta, int tb) {
      const int n = (int)(col / CH), sp = (int)(col % CH);
      const int t_first = std::max(ta - 1, 0);
      for (int t_in = t_first; t_in <= tb; ++t_in) {
        SrStep st;
        st.in_pos = (int32_t)(((int64_t)n * g.TS + t_in + g.ot) * g.SL + (int64_t)sp * 128);
        const int t_out = t_in - 1;
        st.flags = SR_ACTIVE | (t_in == t_first ? SR_FIRST : 0u) | ((t_out >= ta && t_out < tb) ? SR_STORE : 0u) |
                   ((uint32_t)std::min(128, g.SL - sp * 128) << 8);
        lists[sg].push_back(st);
      }
    };
    for (int sg = 0; sg < 2 * grid; ++sg) {
      int64_t g0 = (int64_t)sg * Lr;
      const int64_t g1 = std::min(G, g0 + Lr);
      while (g0 < g1) {
        const int64_t col = g0 / T;
        const int ta = (int)(g0 % T), tb = (int)std::min<int64_t>(T, ta + (g1 - g0));
        add_range(sg, col, ta, tb);
        g0 += tb - ta;
      }
    }
    for (int sg = 0; sg < 2 * grid; ++sg) nsteps = std::max(nsteps, lists[sg].size());
    std::vector<SrStep> flat((size_t)2 * grid * nsteps);
    memset(flat.data(), 0, flat.size() * sizeof(SrStep));
    for (int sg = 0; sg < 2 * grid; ++sg) std::copy(lists[sg].begin(), lists[sg].end(), flat.begin() + (size_t)sg * nsteps);
    lsd_handle::RingTab tab;
    tab.nsteps = (int)nsteps; tab.grid = grid;
    // cache miss only (first forward of a shape): blocking copy, visible to every stream afterwards
    if (cudaMalloc(&tab.dev, std::max<size_t>(flat.size(), 1) * sizeof(SrStep)) != cudaSuccess ||
        cudaMemcpy(tab.dev, flat.data(), flat.size() * sizeof(SrStep), cudaMemcpyHostToDevice) != cudaSuccess)
      return lsd_fail(h, LSD_ERR_CUDA, "stem: step table upload failed");
    it = h->ring_tabs.emplace(key, tab).first;
  }
  *out = &it->second;
  return 0;
}

// Stem through the temporal-ring kernel (stem_ring.cu): xs (pixel rows, 2 parity sets) -> so (plain planar, 64 channels), same geometry.
int run_stem_ring(const BCtx& c, const PBuf& xs, const PBuf& so) {
  lsd_handle* h = c.h;
  const UcGeom& g = xs.g;
  if (g.P_total >= ((int64_t)1 << 31) - 4096) return lsd_fail(h, LSD_ERR_SHAPE, "stem: more than 2^31 padded positions in one launch (reduce the batch)");
  const BLayer& L = h->blayers.at("visual_encoder.stem");
  StemRingP p;
  memset(&p, 0, sizeof(p));
  p.xs[0] = c.org(xs);
  p.xs[1] = c.org(xs) + xs.set_stride;
  p.w = reinterpret_cast<const __nv_bfloat16*>(h->barena) + h->stem_ring_w_off;
  p.bias = h->bbias + L.bias_off;
  p.y = c.org(so);
  p.y_plane_stride = so.plane_stride;
  p.g = g;
  // parity set 0: kernel rows 1, 3, 5 (dh = -1, 0, 1); set 1: rows 0, 2, 4, 6 (dh = -2 .. 1); K chunks are 2-position shifts
  p.ntap[0] = 3; p.ntap[1] = 4;
  for (int t = 0; t < 4; ++t) { p.rel[0][t] = t * g.RW; p.rel[1][t] = t * g.RW; }
  p.start[0] = -g.RW; p.start[1] = -2 * g.RW;
  p.units[0] = 128 + 2 * g.RW + 3; p.units[1] = 128 + 3 * g.RW + 3;
  if ((int64_t)(2 * g.RW + 3) * 8 > xs.origin) return lsd_fail(h, LSD_ERR_UNSUPPORTED, "stem: guard zone too small");
  const lsd_handle::RingTab* tab = nullptr;
  if (int trc = ring_table(c, g, &tab)) return trc;
  p.steps = reinterpret_cast<const SrStep*>(tab->dev);
  p.nsteps = tab->nsteps;
  p.nst = 6;
  if (const char* e = getenv("LSD_SR_SKIP")) p.skip = atoi(e);   // timing experiments only
  while (p.nst > 3 && stem_ring_smem_bytes(p) > 223u * 1024u) --p.nst;    // a long step table (large batches) takes ring stages
  if (stem_ring_smem_bytes(p) > 223u * 1024u) return lsd_fail(h, LSD_ERR_UNSUPPORTED, "stem: batch too large for the ring kernel (LSD_STEM_RING=0)");
  const ConvP& cp = h->convs.at("visual_encoder.stem");
  h->prof.begin(c.st, 2.0 * (double)g.N * g.T * g.H * g.W * 64.0 * (double)cp.kt * cp.kh * cp.kw * cp.Cin, 2);
  if (getenv("LSD_SR_TRACE")) {
    // debug: clock64 stamps of CTA 0, steps 16..47 (producer: stage free / copies issued; MMA slot 0: stage landed / accumulator
    // block free / step issued; epilogue warp 4: accumulator complete / block handed back); prints after a sync
    static long long* dbuf = nullptr;
    constexpr int kDbg = 256 + 4 * 160;
    if (!dbuf) cudaMalloc(&dbuf, kDbg * sizeof(long long));
    cudaMemsetAsync(dbuf, 0, kDbg * sizeof(long long), c.st);
    p.dbg = dbuf;
    launch_stem_ring(p, tab->grid, c.st);
    long long hv[kDbg];
    cudaMemcpyAsync(hv, dbuf, sizeof(hv), cudaMemcpyDeviceToHost, c.st);
    cudaStreamSynchronize(c.st);
    {
      long long g0 = INT64_MAX, g1 = 0, cmin = INT64_MAX, cmax = 0, csum = 0, smax = 0;
      const int nc = std::min(tab->grid, 160);
      for (int i = 0; i < nc; ++i) g0 = std::min(g0, hv[256 + 4 * i]);
      for (int i = 0; i < nc; ++i) {
        const long long* d = hv + 256 + 4 * i;
        g1 = std::max(g1, d[1]); smax = std::max(smax, d[0] - g0);
        const long long cy = d[3] - d[2];
        cmin = std::min(cmin, cy); cmax = std::max(cmax, cy); csum += cy;
      }
      fprintf(stderr, "[sr] %d CTAs x %d steps: kernel span %.1f us (globaltimer), latest CTA start +%.1f us, CTA cycles min %lld avg %lld max %lld\n", nc,
              p.nsteps, (g1 - g0) / 1e3, smax / 1e3, cmin, csum / nc, cmax);
    }
    const long long t0 = hv[0];
    for (int k = 0; k < 32; ++k)
      fprintf(stderr, "[sr] step %2d | prod free %7lld issued %7lld | mma landed %7lld blockfree %7lld issued %7lld | epi complete %7lld back %7lld\n", k + 16,
              hv[(0 * 32 + k) * 2] - t0, hv[(0 * 32 + k) * 2 + 1] - t0, hv[(1 * 32 + k) * 2] - t0, hv[(1 * 32 + k) * 2 + 1] - t0,
              hv[(2 * 32 + k) * 2] - t0, hv[(3 * 32 + k) * 2] - t0, hv[(3 * 32 + k) * 2 + 1] - t0);
    h->prof.end(c.st);
    return 0;
  }
  launch_stem_ring(p, tab->grid, c.st);
  h->prof.end(c.st);
  return 0;
}

#define RUN(name, ...)                            \
  do {                                            \
    UArgs a_;                                     \
    __VA_ARGS__;                                  \
    if ((rc = run_umma(b, name, a_))) return rc;  \
  } while (0)

#define RUNC(ctx, name, ...)                        \
  do {                                              \
    UArgs a_;                                       \
    __VA_ARGS__;                                    \
    if ((rc = run_umma(ctx, name, a_))) return rc;  \
  } while (0)

#define RUNS(name, ...)                            \
  do {                                             \
    UArgs a_;                                      \
    __VA_ARGS__;                                   \
    if ((rc = run_umma(bs, name, a_))) return rc;  \
  } while (0)

PlanarOut pout(const BCtx& c, const PBuf& p, const PBuf* lo = nullptr, int plane_off = 0) {
  PlanarOut o;
  o.y = c.org(p) + (int64_t)plane_off * p.plane_stride;
  o.ylo = lo ? c.org(*lo) + (int64_t)plane_off * lo->plane_stride : nullptr;
  o.plane_stride = p.plane_stride;
  if (p.g.ow > 0 && p.g.HP == 1) { o.grp = p.g.W; o.grp_stride = p.g.RW; o.off = p.g.ow; }   // padded token geometry
  else { o.grp = 0; o.grp_stride = 0; o.off = 0; }                                            // plain rows
  return o;
}

// Residual stage: conv1 (+ReLU) -> conv2 (+fused strided 1x1 downsample | +identity) -> ReLU
int res_stage_umma(const BCtx& b, const std::string& p, const PBuf& x, const PBuf& mid, const PBuf& y, bool has_ds, int y_mode,
                   const PBuf* x_lo = nullptr, const PBuf* mid_lo = nullptr, const PBuf* y_lo = nullptr) {
  int rc = 0;
  RUN(p + ".conv1", a_.in = &x; a_.in_lo = x_lo; a_.og = mid.g; a_.act = ACT_RELU; a_.yp = &mid; a_.yp_lo = mid_lo);
  if (has_ds) RUN(p + ".conv2", a_.in = &mid; a_.in_lo = mid_lo; a_.in_ds = &x; a_.in_ds_lo = x_lo; a_.og = mid.g; a_.act = ACT_RELU;
                  a_.yp = &y; a_.yp_lo = y_lo; a_.y_mode = y_mode);
  else RUN(p + ".conv2", a_.in = &mid; a_.in_lo = mid_lo; a_.og = mid.g; a_.act = ACT_RELU; a_.yp = &y; a_.yp_lo = y_lo; a_.y_mode = y_mode;
           a_.res = &x; a_.res_lo = x_lo);
  return 0;
}

// One folded small-map convolution (UcFoldSlice in umma_conv.cuh) of layer `name` (weights "<name>#fold"): x holds the input map
// (Hi x Wi, one plane set per position, row geometry), read with stride `stride`; x_ds (optional) is the input of the fused 1x1
// stride-2 downsample (map Hd x Wd).  Output map Ho x Wo, ReLU, to yp: folded (UC_Y_FOLD) or a plain padded map (UC_Y_MAP).
int run_umma_fold(const BCtx& c, const std::string& name, const PBuf& x, int Hi, int Wi, int stride, const PBuf* x_ds, int Hd, int Wd,
                  int Ho, int Wo, const PBuf& yp, int y_mode) {
  const auto itL = c.h->blayers.find(name + "#fold");
  if (itL == c.h->blayers.end()) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: no weights packed for the folded route (LSD_FOLD=0)", name.c_str());
  const BLayer& L = itL->second;
  const UcGeom& og = x.g;   // row geometry: the tile positions are frame rows
  if (og.P_total >= ((int64_t)1 << 31) - 1024) return lsd_fail(c.h, LSD_ERR_SHAPE, "%s: more than 2^31 rows in one launch (reduce the batch)", name.c_str());
  if ((L.groups.size() == 2) != (x_ds != nullptr) || x.sets != Hi * Wi || (x_ds && x_ds->sets != Hd * Wd))
    return lsd_fail(c.h, LSD_ERR_ARG, "%s: folded inputs do not match the layer", name.c_str());
  UmmaConvP p;
  memset(&p, 0, sizeof(p));
  p.w = reinterpret_cast<const __nv_bfloat16*>(c.h->barena);
  p.bias = c.h->bbias + L.bias_off;
  p.Cout = L.ntile;
  p.act = ACT_RELU;
  p.g = og;
  p.fold = 1;
  p.y_mode = y_mode;
  p.y = c.org(yp);
  p.y_plane_stride = yp.plane_stride; p.y_set_stride = yp.set_stride;
  p.g2 = yp.g;
  p.ymap_W = Wo;
  // Tile shape: 2 M-tiles x 128 columns (LSD_FOLD_MT / LSD_FOLD_NT: tuning knobs), fewer M-tiles when the rows do not fill them.
  // One tile per CTA: slices differ in K (4 / 6 / 9 input positions for corner / edge / centre), the heaviest come first and the
  // block scheduler hands the rest to the SMs as they free up.
  int mt = 2;
  if (const char* e = LSD_ENV("LSD_FOLD_MT")) mt = std::max(1, std::min(4, atoi(e)));
  p.MT = (int)std::max<int64_t>(1, std::min<int64_t>(mt, (og.P_total + 127) / 128));
  p.nbuf = 1;
  p.issuers = std::min(p.MT, 4);
  uint32_t cols = 32;
  while ((int)cols < p.MT * L.ntile) cols *= 2;
  p.tmem_cols = cols;
  const int S = p.MT * 128;
  const PBuf* srcs[2] = {&x, x_ds};
  p.ngroups = (int)L.groups.size();
  p.nbands = p.ngroups;
  int max_a = 0, max_w = 0, min_k16 = 1 << 30;
  for (int gi = 0; gi < p.ngroups; ++gi) {
    const BGroup& G = L.groups[gi];
    UcGroup& ug = p.groups[gi];
    ug.band_begin = gi; ug.band_end = gi + 1;
    ug.k16 = G.k16; ug.taps_total = G.taps_total;
    ug.w_off = (int64_t)G.w_off; ug.slice_stride = (int64_t)G.slice_stride;
    // launch-wide band shapes the MMA issuer reads: main = 3 temporal taps (rows -1, 0, +1), downsample = 1 tap (row 0); each
    // stage's A source (plane set of one input position) is baked into the slice programs below
    UcBand& ub = p.bands[gi];
    const PBuf& src = *srcs[gi];
    ub.base = c.org(src);
    ub.plane_stride = src.plane_stride;
    ub.chunk_stride = 2 * src.plane_stride;
    ub.ntaps = gi == 0 ? 3 : 1;
    ub.start = gi == 0 ? -1 : 0;
    ub.len_extra = gi == 0 ? 2 : 0;
    for (int j = 0; j < ub.ntaps; ++j) ub.rel[j] = j;
    if ((int64_t)8 > src.origin) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: guard zone too small", name.c_str());
    max_a = std::max(max_a, 2 * (S + ub.len_extra) * 16);
    max_w = std::max(max_w, ub.ntaps * L.ntile * 32);
    min_k16 = std::min(min_k16, G.k16);
  }
  // K chunks per stage: the summation order (input position, K chunk, temporal tap) does not depend on kpack here, so the stages
  // can be large enough to amortise the per-stage bookkeeping of the issuing warps
  p.kpack = std::max(1, std::min(std::min(8, min_k16), (48 * 1024) / (max_a + max_w)));
  p.a_stage_bytes = ((uint32_t)(max_a * p.kpack) + 127u) & ~127u;
  p.w_stage_bytes = (uint32_t)(max_w * p.kpack);
  // column slices: (output position, Cout slice), heaviest positions first
  const int cslices = L.Cout / L.ntile;
  std::vector<std::array<int, 3>> pos;   // (-in-bounds input positions, ho, wo)
  auto inb = [&](int o, int k, int n) { const int i = stride * o + k - 1; return i >= 0 && i < n; };
  for (int ho = 0; ho < Ho; ++ho)
    for (int wo = 0; wo < Wo; ++wo) {
      int nq = 0;
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) nq += inb(ho, kh, Hi) && inb(wo, kw, Wi);
      pos.push_back({-nq, ho, wo});
    }
  std::stable_sort(pos.begin(), pos.end(), [](const std::array<int, 3>& a, const std::array<int, 3>& b) { return a[0] < b[0]; });
  const int nslices = (int)pos.size() * cslices;
  if (nslices > UC_MAX_FSLICES || Ho > 255 || Wo > 255) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: map too large for the folded route", name.c_str());
  auto chunks = [&](int k16) { return (k16 + p.kpack - 1) / p.kpack; };
  int off = 0;
  for (int i = 0; i < nslices; ++i) {
    const auto& q = pos[(size_t)(i / cslices)];
    const int nst = -q[0] * chunks(p.groups[0].k16) + (x_ds ? chunks(p.groups[1].k16) : 0);
    p.fslice[i] = UcFoldSlice{(uint16_t)off, (uint16_t)nst, (uint8_t)q[1], (uint8_t)q[2], (uint8_t)(i % cslices), 0};
    p.nst_tile = std::max(p.nst_tile, nst);
    off += nst;
  }
  if (off > 65535) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: folded stage programs too long", name.c_str());
  const uint32_t stage = p.a_stage_bytes + p.w_stage_bytes;
  const uint32_t prog_bytes = (uint32_t)p.nst_tile * (uint32_t)umma_conv_stage_desc_bytes();
  const uint32_t budget = 211u * 1024u - (uint32_t)umma_conv_extra_smem_bytes(p);
  if (prog_bytes + 2 * stage > budget) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: stage program of %u bytes does not fit", name.c_str(), prog_bytes);
  p.stages = std::max(2, std::min((int)((budget - prog_bytes) / stage), 8));
  if (const char* e = getenv("LSD_UMMA_SKIP")) p.skip = atoi(e);
  if (const char* why = umma_conv_config_error(p)) return lsd_fail(c.h, LSD_ERR_UNSUPPORTED, "%s: %s", name.c_str(), why);
  // slice programs: per in-bounds input position q (ascending), per K-chunk block, one stage of 3 temporal taps with A from plane
  // set q; then the downsample (input position (2 ho, 2 wo)).  Summation order (q, K chunk, dt): fixed by the geometry alone.
  auto build = [&](std::vector<UcStageDesc>& v) {
    for (int i = 0; i < nslices; ++i) {
      const UcFoldSlice& f = p.fslice[i];
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) {
          if (!inb(f.h, kh, Hi) || !inb(f.w, kw, Wi)) continue;
          UcBand bq = p.bands[0];
          bq.base = c.org(x) + (int64_t)((stride * f.h + kh - 1) * Wi + stride * f.w + kw - 1) * x.set_stride;
          bq.tap_begin = (kh * 3 + kw) * 3;   // (kh, kw, kt) packing order, see Packer::add_fold
          for (int c0 = 0; c0 < p.groups[0].k16; c0 += p.kpack) v.push_back(umma_conv_stage(p, p.groups[0], bq, 0, c0, f.col));
        }
      if (x_ds) {
        UcBand bd = p.bands[1];
        bd.base = c.org(*x_ds) + (int64_t)(2 * f.h * Wd + 2 * f.w) * x_ds->set_stride;
        for (int c0 = 0; c0 < p.groups[1].k16; c0 += p.kpack) v.push_back(umma_conv_stage(p, p.groups[1], bd, 1, c0, f.col));
      }
    }
  };
  if (int rc = stage_program(c, name + "#fold", p, build, {(uint64_t)Hi, (uint64_t)Wi, (uint64_t)stride, (uint64_t)Hd, (uint64_t)Wd,
                                                          (uint64_t)x.set_stride, (uint64_t)(x_ds ? x_ds->set_stride : 0)})) return rc;
  // profile FLOPs: the algorithmic count of the original convolution (the row geometry has H = W = 1)
  double kflop = 0;
  for (const BGroup& G : L.groups) kflop += (double)G.taps_total * G.Cin;
  c.h->prof.begin(c.st, 2.0 * (double)og.N * og.T * Ho * Wo * L.Cout * kflop, 2);
  launch_umma_conv(p, nslices, c.st, c.h->num_sms, c.max_ctas);
  c.h->prof.end(c.st);
  return 0;
}

// Residual stage with a stride-2 conv1 and a fused downsample on the folded route: x (folded, Hi x Wi) -> mid (folded, Ho x Wo)
// -> y (folded, or the plain padded map when y_mode == UC_Y_MAP)
int res_stage_fold(const BCtx& b, const std::string& p, const PBuf& x, int Hi, int Wi, const PBuf& mid, int Ho, int Wo, const PBuf& y, int y_mode) {
  int rc = 0;
  if ((rc = run_umma_fold(b, p + ".conv1", x, Hi, Wi, 2, nullptr, 0, 0, Ho, Wo, mid, UC_Y_FOLD))) return rc;
  return run_umma_fold(b, p + ".conv2", mid, Ho, Wo, 1, &x, Hi, Wi, Ho, Wo, y, y_mode);
}

}  // namespace

// Weight stream, stage table and small vectors of the fused temporal-transformer kernel (tok_fused.cu).
static int pack_tok_fused(lsd_handle* h, const std::vector<float>& f32) {
  std::vector<TfBlock> blocks;
  tf_layer_blocks(blocks);
  std::vector<uint32_t> stage_bytes;
  for (const TfBlock& b : blocks)
    for (int k0 = 0; k0 < b.k16; k0 += b.kps) stage_bytes.push_back((uint32_t)b.kps * (uint32_t)b.N * 32u);
  std::vector<__half> w;
  std::vector<float> vec((size_t)TF_LAYERS * TF_VEC_LAYER + (size_t)(2 * TF_LAYERS + 1) * TF_D, 0.f);
  std::vector<float> cum(TF_D, 0.f);
  float* cum_out = vec.data() + (size_t)TF_LAYERS * TF_VEC_LAYER;
  for (int l = 0; l < TF_LAYERS; ++l) {
    const std::string k = "t" + std::to_string(l);
    const ConvP &cin = h->convs.at(k + ".in"), &cout = h->convs.at(k + ".out"), &cf1 = h->convs.at(k + ".ff1"), &cf2 = h->convs.at(k + ".ff2");
    const size_t w0 = w.size();
    for (const TfBlock& b : blocks) {
      const ConvP& c = b.kind == 0 ? cin : (b.kind == 1 ? cout : (b.kind == 2 ? cf1 : cf2));
      for (int k16 = 0; k16 < b.k16; ++k16)
        for (int pl = 0; pl < 2; ++pl)
          for (int n = 0; n < b.N; ++n)
            for (int e = 0; e < 8; ++e) {
              const int kk = k16 * 16 + pl * 8 + e;
              int co, ci;
              if (b.kind == 0) { co = ((n % 96) / 32) * 256 + (2 * b.idx + n / 96) * 32 + (n % 32); ci = kk; }
              else if (b.kind == 1) { co = n; ci = 64 * b.idx + kk; }
              else if (b.kind == 2) { co = 128 * b.idx + n; ci = kk; }
              else { co = n; ci = 128 * b.idx + kk; }
              w.push_back(__float2half_rn(f32[c.w_off + (size_t)ci * c.Cout + co]));
            }
    }
    if (l == 0) h->tokf_layer_bytes = (uint32_t)((w.size() - w0) * sizeof(__half));
    float* lv = vec.data() + (size_t)l * TF_VEC_LAYER;
    const char* names[4] = {".ln1.w", ".ln1.b", ".ln2.w", ".ln2.b"};
    for (int i = 0; i < 4; ++i) memcpy(lv + 256 * i, &f32[h->vecs.at(k + names[i])], 256 * sizeof(float));
    for (int n = 0; n < 768; ++n) {   // packed order: [head pair][head in pair][Q|K|V][32]
      const int hp = n / 192, r = n % 192;
      lv[1024 + n] = f32[cin.shift_off + ((r % 96) / 32) * 256 + (2 * hp + r / 96) * 32 + (r % 32)];
    }
    memcpy(lv + 1024 + 768, &f32[cf1.shift_off], 1024 * sizeof(float));
    // cumulative biases of the GEMMs that accumulate straight into the residual stream
    memcpy(cum_out + (size_t)(2 * l) * TF_D, cum.data(), TF_D * sizeof(float));
    for (int i = 0; i < TF_D; ++i) cum[i] += f32[cout.shift_off + i];
    memcpy(cum_out + (size_t)(2 * l + 1) * TF_D, cum.data(), TF_D * sizeof(float));
    for (int i = 0; i < TF_D; ++i) cum[i] += f32[cf2.shift_off + i];
  }
  memcpy(cum_out + (size_t)(2 * TF_LAYERS) * TF_D, cum.data(), TF_D * sizeof(float));
  h->tokf_n_stage = (int)stage_bytes.size();
  for (void* q : {(void*)h->tokf_w, (void*)h->tokf_stage_bytes, (void*)h->tokf_vec}) if (q) cudaFree(q);
  h->tokf_w = nullptr; h->tokf_stage_bytes = nullptr; h->tokf_vec = nullptr;
  cudaError_t e = cudaMalloc(&h->tokf_w, w.size() * sizeof(__half));
  if (e == cudaSuccess) e = cudaMemcpy(h->tokf_w, w.data(), w.size() * sizeof(__half), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc(&h->tokf_stage_bytes, stage_bytes.size() * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMemcpy(h->tokf_stage_bytes, stage_bytes.data(), stage_bytes.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc(&h->tokf_vec, vec.size() * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(h->tokf_vec, vec.data(), vec.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return lsd_fail(h, LSD_ERR_CUDA, "pack_tok_fused: %s", cudaGetErrorString(e));
  return 0;
}

// Weight stream and vectors of the fused token-path front (tok_front.cu), in the order of tok_front.cuh.
static int pack_tok_front(lsd_handle* h, const std::vector<float>& f32) {
  std::vector<__half> w;
  w.reserve((size_t)TFR_K16_TOTAL * 16 * 256);
  // one (256 x 16*k16) block, packed [k16][2 planes][256][8]; get(ci, co) = weight of input channel ci, output channel co
  auto emit = [&](int k16, auto&& get) {
    for (int k = 0; k < k16; ++k)
      for (int pl = 0; pl < 2; ++pl)
        for (int n = 0; n < 256; ++n)
          for (int e = 0; e < 8; ++e) w.push_back(__float2half_rn(get(k * 16 + pl * 8 + e, n)));
  };
  const ConvP &o0 = h->convs.at("cross.v2a.out"), &o1 = h->convs.at("cross.a2v.out"), &g0 = h->convs.at("cross.gate0"),
              &fu = h->convs.at("cross.fuse"), &pp = h->convs.at("temporal.pre_scale_proj");
  for (const ConvP* o : {&o0, &o1})
    for (int hp = 0; hp < 4; ++hp) emit(4, [&](int ci, int co) { return f32[o->w_off + (size_t)(64 * hp + ci) * 256 + co]; });
  emit(32, [&](int ci, int co) { return f32[g0.w_off + (size_t)ci * 256 + co]; });
  emit(16, [&](int ci, int co) { return f32[fu.w_off + (size_t)ci * 256 + co]; });
  const int ks[3] = {3, 5, 7};
  for (int b = 0; b < 3; ++b) {
    const ConvP& c = h->convs.at("temporal.branch_k" + std::to_string(ks[b]));
    for (int j = 0; j < ks[b]; ++j)     // BN scale folded into the weights, shift added in the epilogue
      emit(16, [&](int ci, int co) { return f32[c.w_off + ((size_t)j * 256 + ci) * 256 + co] * (c.has_scale ? f32[c.scale_off + co] : 1.0f); });
    emit(16, [&](int ci, int co) { return f32[pp.w_off + (size_t)(256 * b + ci) * 256 + co]; });
  }
  if (w.size() != (size_t)TFR_N_STAGES * TFR_STAGE_BYTES / sizeof(__half)) return lsd_fail(h, LSD_ERR_WEIGHTS, "pack_tok_front: stream size mismatch");
  std::vector<float> vec(TFR_V_TOTAL, 0.f);
  auto cp = [&](int dst, size_t src, int n) { memcpy(vec.data() + dst, &f32[src], (size_t)n * sizeof(float)); };
  cp(TFR_V_BO0, o0.shift_off, 256); cp(TFR_V_BO1, o1.shift_off, 256); cp(TFR_V_BG0, g0.shift_off, 256);
  cp(TFR_V_WG2, h->vecs.at("cross.gate2.w"), 256); cp(TFR_V_BG2, h->vecs.at("cross.gate2.b"), 1);
  cp(TFR_V_BF, fu.shift_off, 256);
  cp(TFR_V_SH3, h->convs.at("temporal.branch_k3").shift_off, 256); cp(TFR_V_SH5, h->convs.at("temporal.branch_k5").shift_off, 256);
  cp(TFR_V_SH7, h->convs.at("temporal.branch_k7").shift_off, 256);
  cp(TFR_V_BP, pp.shift_off, 256); cp(TFR_V_CLS, h->vecs.at("temporal.cls"), 256);
  for (void* q : {(void*)h->tokfr_w, (void*)h->tokfr_vec}) if (q) cudaFree(q);
  h->tokfr_w = nullptr; h->tokfr_vec = nullptr;
  cudaError_t e = cudaMalloc(&h->tokfr_w, w.size() * sizeof(__half));
  if (e == cudaSuccess) e = cudaMemcpy(h->tokfr_w, w.data(), w.size() * sizeof(__half), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc(&h->tokfr_vec, vec.size() * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(h->tokfr_vec, vec.data(), vec.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return lsd_fail(h, LSD_ERR_CUDA, "pack_tok_front: %s", cudaGetErrorString(e));
  return 0;
}

int pack_bf16_weights(lsd_handle* h, const std::vector<float>& f32_arena) {
  Packer P{h, f32_arena, {}, {}};
  memcpy(h->lapw_host, &f32_arena[h->convs.at("art.lap").w_off], sizeof(h->lapw_host));   // (video_rows takes them by value)
  h->blayers.clear();
  const int vstr[4] = {1, 2, 2, 2};
  for (int l = 1; l <= 4; ++l) {
    const std::string p = "visual_encoder.layer" + std::to_string(l);
    const int s = vstr[l - 1];
    // Cout slice width per CTA (0 = all columns).  256-column layers run as two 128-column slices: a 128-column stage carries
    // twice the MMA time per refill (4 M-tiles per weight stage instead of 2), measured 15-18 % faster than one 256-column slice.
    int nt = l >= 3 ? 128 : 0;
    if (const char* e = getenv(l == 3 ? "LSD_UMMA_NT3" : (l == 4 ? "LSD_UMMA_NT4" : "LSD_UMMA_NTX"))) nt = atoi(e);   // tuning knob
    // CTA pairs (cta_group::2) for the Cout = 64 layers — stem and layer1, bound by the shared-memory read port
    const bool pairs = l == 1;
    P.add(p + ".conv1", p + ".conv1", s, s, "", nt, false, /*merge_kt=*/l >= 2, pairs);   // 12x12 / 6x6 / 3x3 maps: one band per parity set
    P.ds_sh = 2; P.ds_sw = 2;
    P.add(p + ".conv2", p + ".conv2", 1, 1, l == 1 ? "" : p + ".downsample", nt, false, false, pairs);
    if (l >= 3) {   // folded small-map route (run_umma_fold)
      int fnt = 128;
      if (const char* e = LSD_ENV("LSD_FOLD_NT")) fnt = atoi(e) == 256 ? 256 : 128;   // tuning knob: columns per folded CTA
      P.add_fold(p + ".conv1#fold", p + ".conv1", "", fnt);
      P.add_fold(p + ".conv2#fold", p + ".conv2", p + ".downsample", fnt);
    }
  }
  P.add_toeplitz("visual_encoder.stem", "visual_encoder.stem", 8, 0, false, true);  // 7 taps in w -> 8-pixel window starting at 2*wo-4
  {
    // the same weights for the temporal-ring kernel (stem_ring.cu): per (parity set, kernel row) tap and K chunk one block
    // [2 K halves][192 = 3 temporal taps x 64 columns][8]; column block j holds the weights of temporal tap dt = j - 1
    const ConvP& c = h->convs.at("visual_encoder.stem");
    h->stem_ring_w_off = 0;
    if (c.kt == 3 && c.kh == 7 && c.kw == 7 && c.Cin == 3 && c.Cout == 64) {
      h->stem_ring_w_off = P.w.size();
      const float* W = &f32_arena[c.w_off];
      const float* sc = c.has_scale ? &f32_arena[c.scale_off] : nullptr;
      for (int set = 0; set < 2; ++set)
        for (int b = 0; b < 7; ++b) {
          if (((b - 3) & 1) != set) continue;          // rows of this parity set, in ascending dh
          for (int ch = 0; ch < 2; ++ch)
            for (int kc = 0; kc < 2; ++kc)
              for (int n = 0; n < 192; ++n)
                for (int e = 0; e < 8; ++e) {
                  const int k = ch * 16 + kc * 8 + e, j = k / 4, kw = j - 1, ci = k % 4, a = n / 64, co = n % 64;
                  float v = 0.f;
                  if (ci < 3 && kw >= 0 && kw < 7) v = W[((size_t)((a * 7 + b) * 7 + kw) * 3 + ci) * 64 + co] * (sc ? sc[co] : 1.0f);
                  P.w.push_back(f2bf(v));
                }
        }
      while (P.w.size() % 64) P.w.push_back(0);
    }
  }
  P.add_toeplitz("art.hf0", "art.hf0", 4, 1);                          // 3 taps in w -> 4-pixel window starting at 2*wo-2
  P.add("art.td0", "art.td0", 1, 1);
  P.add("art.td3", "art.td3", 1, 1);
  P.add("art.hf3", "art.hf3", 2, 2);
  // audio encoder (audio_encoder.py:128-156): strides (1,1), (2,2), (2,1), (2,1)
  P.add_toeplitz("audio_encoder.stem", "audio_encoder.stem", 8, 0, true);
  const int ash[4] = {1, 2, 2, 2}, asw[4] = {1, 2, 1, 1};
  for (int l = 1; l <= 4; ++l) {
    const std::string p = "audio_encoder.layer" + std::to_string(l);
    // split-bf16: the audio encoder is 1.4 % of the FLOPs but its bf16 rounding dominated the logit error
    P.add(p + ".conv1", p + ".conv1", ash[l - 1], asw[l - 1], "", 0, true);
    P.ds_sh = ash[l - 1]; P.ds_sw = asw[l - 1];
    P.add(p + ".conv2", p + ".conv2", 1, 1, l == 1 ? "" : p + ".downsample", 0, true);
  }
  // token path GEMMs: 64-column slices so that the small M (B*T rows) still spreads over the SMs; the wide ones (768 / 1024
  // columns) use 128-column slices, which keeps B = 64 (17 M-tiles) inside one wave of CTAs
  int wide = 128;
  if (const char* e = LSD_ENV("LSD_UMMA_NTW")) wide = atoi(e);   // tuning knob
  int narrow = 64;
  if (const char* e = LSD_ENV("LSD_UMMA_NTN")) narrow = atoi(e);   // tuning knob
  for (const char* k : {"projection.visual_proj", "projection.audio_proj", "cross.v2a.out", "cross.a2v.out",
                        "cross.gate0", "cross.fuse", "temporal.branch_k3", "temporal.branch_k5", "temporal.branch_k7",
                        "temporal.pre_scale_proj"})
    P.add_split(k, k, narrow);
  for (const char* k : {"cross.in_v", "cross.in_a", "cross.vcomb", "cross.acomb"}) P.add_split(k, k, wide);
  for (int l = 0; l < 4; ++l)
    for (const char* k : {".in", ".out", ".ff1", ".ff2"})
      P.add_split("t" + std::to_string(l) + k, "t" + std::to_string(l) + k, (k[1] == 'i' || (k[1] == 'f' && k[3] == '1')) ? wide : narrow);
  if (h->barena) { cudaFree(h->barena); h->barena = nullptr; }
  if (h->bbias) { cudaFree(h->bbias); h->bbias = nullptr; }
  cudaError_t e = cudaMalloc(&h->barena, P.w.size() * 2);
  if (e == cudaSuccess) e = cudaMemcpy(h->barena, P.w.data(), P.w.size() * 2, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc(&h->bbias, P.bias.size() * 4);
  if (e == cudaSuccess) e = cudaMemcpy(h->bbias, P.bias.data(), P.bias.size() * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return lsd_fail(h, LSD_ERR_CUDA, "pack_bf16_weights: %s", cudaGetErrorString(e));
  if (int rc = pack_tok_fused(h, f32_arena)) return rc;
  return pack_tok_front(h, f32_arena);
}

void make_plan_bf16(lsd_handle* h, int B, int T, int H, int W, int F, int Ta, std::vector<Stage>& stages, size_t& bytes) {
  Shapes s;
  if (make_shapes(h, B, T, H, W, F, Ta, s) != 0) { bytes = 0; return; }
  BPlan P;
  build_plan(s, P);
  stages = P.f32.stages;
  bytes = P.f32.cursor;
}

// Debug timeline (LSD_TIMELINE=1, never in timed runs): timestamps of the phases of one forward on all of its streams, relative to
// the start of the forward; printed to stderr after a device synchronisation.
struct Timeline {
  bool on = false;
  std::vector<std::pair<std::string, cudaEvent_t>> marks;
  void mark(cudaStream_t st, const char* name) {
    if (!on) return;
    cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st);
    marks.emplace_back(name, e);
  }
  void dump() {
    if (!on || marks.empty()) return;
    cudaDeviceSynchronize();
    fprintf(stderr, "[timeline]");
    for (auto& m : marks) { float ms = 0; cudaEventElapsedTime(&ms, marks[0].second, m.second); fprintf(stderr, " %s=%.0f", m.first.c_str(), ms * 1000.0f); }
    fprintf(stderr, " (us)\n");
    for (auto& m : marks) cudaEventDestroy(m.second);
    marks.clear();
  }
};
static Timeline g_tl;

// AudioEncoder.forward (audio_encoder.py:173-205) on tcgen05: log-mel windows -> a_feat (B, A4, 256) fp32 + planar (hi, lo) copy
static int audio_encoder_bf16(const BCtx& b, const Shapes& s, bool inputs_ready, const void* audio, int adt) {
  const BPlan& P = *b.P;
  auto pbf = [&](const char* n) -> const PBuf& { return P.pb.at(n); };
  cudaStream_t st = b.st;
  int rc = 0;
  // ---- audio encoder (audio_encoder.py:173-205) on tcgen05
  const PBuf &xa = pbf("xa"), &sao = pbf("sa_out"), &a1 = pbf("a1");
  if (inputs_ready) launch_audio_rows(b.f("aud"), LSD_F32, b.org(xa), xa.set_stride, xa.g, s.F, s.Ta, st);
  else launch_audio_rows(audio, adt, b.org(xa), xa.set_stride, xa.g, s.F, s.Ta, st);
  RUN("audio_encoder.stem", a_.in = &xa; a_.og = xa.g; a_.act = ACT_RELU; a_.yp = &sao; a_.yp_lo = &pbf("sa_out_lo"));
  launch_planar_maxpool(b.org(sao), sao.plane_stride, sao.g, b.org(a1), a1.plane_stride, a1.g, 64, st, b.org(pbf("sa_out_lo")), b.org(pbf("a1_lo")));
  if ((rc = res_stage_umma(b, "audio_encoder.layer1", a1, pbf("a1a"), pbf("ya1"), false, UC_Y_PARITY, &pbf("a1_lo"), &pbf("a1a_lo"), &pbf("ya1_lo")))) return rc;
  if ((rc = res_stage_umma(b, "audio_encoder.layer2", pbf("ya1"), pbf("a2a"), pbf("ya2"), true, UC_Y_PARITY_H, &pbf("ya1_lo"), &pbf("a2a_lo"), &pbf("ya2_lo")))) return rc;
  if ((rc = res_stage_umma(b, "audio_encoder.layer3", pbf("ya2"), pbf("a3a"), pbf("ya3"), true, UC_Y_PARITY_H, &pbf("ya2_lo"), &pbf("a3a_lo"), &pbf("ya3_lo")))) return rc;
  if ((rc = res_stage_umma(b, "audio_encoder.layer4", pbf("ya3"), pbf("a4a"), pbf("ya4"), true, UC_Y_PLAIN, &pbf("ya3_lo"), &pbf("a4a_lo"), &pbf("ya4_lo")))) return rc;
  const PBuf& ya4 = pbf("ya4");
  launch_planar_mean2(b.org(ya4), ya4.plane_stride, ya4.g, 256, b.f("a_feat"), 256, 2, pout(b, pbf("afeat_p"), &pbf("afeat_p_lo")), st,
                      b.org(pbf("ya4_lo")));  // mean over F'
  return 0;
}

// CrossModalAttention.forward + TemporalTransformer.forward (fusion_module.py:54-87, temporal.py:79-111): expects v_emb / a_emb
// (fp32 rows) and vemb_p (planar hi, lo) in the workspace; leaves the fused tokens in "fused" and the transformer tokens in "tok".
// combined: "vcomb" / "acomb" already hold [emb | in-projection] of the visual / interpolated audio tokens (full forward with the
// fused front kernel); otherwise v_emb / a_emb (+ vemb_p) are the inputs and the in-projections are computed here.
static bool token_front_enabled(int T) {
  const char* e = getenv("LSD_TOK_FRONT");
  return !(e && atoi(e) == 0) && tok_front_supported(T);
}
// vcomb / K (shared-visual forward): the merged visual projection lives in another workspace, window w reads its row group w / K.
static int token_path_bf16(const BCtx& b, const Shapes& s, bool combined = false, const float* vcomb = nullptr, int K = 1) {
  const BPlan& P = *b.P;
  auto pbf = [&](const char* n) -> const PBuf& { return P.pb.at(n); };
  cudaStream_t st = b.st;
  const int B = s.B, T = s.T, TA = s.A4, NT = T + 1;
  const UcGeom gt = P.gt;
  int rc = 0;
  // Independent pieces run side by side on two helper streams: the token path is a chain of latency-bound launches, each far too
  // small to fill the SMs it gets.
  lsd_handle* h = b.h;
  if (!h->tok_stream[0]) {
    for (int i = 0; i < 2; ++i)
      if (cudaStreamCreateWithFlags(&h->tok_stream[i], cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&h->ev_tok_join[i], cudaEventDisableTiming) != cudaSuccess)
        return lsd_fail(h, LSD_ERR_CUDA, "token helper stream creation failed");
    if (cudaEventCreateWithFlags(&h->ev_tok_fork, cudaEventDisableTiming) != cudaSuccess) return lsd_fail(h, LSD_ERR_CUDA, "token helper event creation failed");
  }
  BCtx b1 = b, b2 = b;                      // helper-stream contexts (same workspace and plan)
  b1.st = h->tok_stream[0]; b2.st = h->tok_stream[1];
  auto fork = [&](int n) { cudaEventRecord(h->ev_tok_fork, st); for (int i = 0; i < n; ++i) cudaStreamWaitEvent(h->tok_stream[i], h->ev_tok_fork, 0); };
  auto join = [&](int n) { for (int i = 0; i < n; ++i) { cudaEventRecord(h->ev_tok_join[i], h->tok_stream[i]); cudaStreamWaitEvent(st, h->ev_tok_join[i], 0); } };
  // ---- cross-modal attention + gated fusion (fusion_module.py:54-87)
  float *pv = combined ? nullptr : b.f("proj_v"), *pa = combined ? nullptr : b.f("proj_a"), *gi = b.f("gate_in");   // (combined: tok_front reads vcomb / acomb)
  if (!combined) {
    fork(1);
    launch_lerp_tokens_p(b.f("a_emb"), b.f("a_int"), B, TA, T, 256, pout(b, pbf("aint_p"), &pbf("aint_p_lo")), b1.st);
    RUNC(b1, "cross.in_a", a_.in = &pbf("aint_p"); a_.in_lo = &pbf("aint_p_lo"); a_.og = gt; a_.y32 = pa; a_.y32_ld = 768);
    RUN("cross.in_v", a_.in = &pbf("vemb_p"); a_.in_lo = &pbf("vemb_p_lo"); a_.og = gt; a_.y32 = pv; a_.y32_ld = 768);
    join(1);
  }
  g_tl.mark(st, "T:inproj");
  float* tok = b.f("tok");
  // ---- attention core, output projections, gated fusion, multi-scale branches, pre_scale_proj, CLS row: one fused launch
  // (tok_front.cu); LSD_TOK_FRONT=0 (debug / A-B tests) or more than 61 tokens per window fall back to the launch-by-launch chain
  if (token_front_enabled(T)) {
    TokFrontP fp;
    memset(&fp, 0, sizeof(fp));
    if (combined) {
      fp.v_emb = vcomb ? vcomb : b.f("vcomb"); fp.pv = fp.v_emb + 256; fp.a_int = b.f("acomb"); fp.pa = fp.a_int + 256;
      fp.ld_e = 1024; fp.ld_p = 1024;
    } else {
      fp.pv = pv; fp.pa = pa; fp.v_emb = b.f("v_emb"); fp.a_int = b.f("a_int");
      fp.ld_e = 256; fp.ld_p = 768;
    }
    fp.gi = gi; fp.fused = b.f("fused"); fp.tok = tok;
    fp.w = reinterpret_cast<const __half*>(h->tokfr_w);
    fp.vec = h->tokfr_vec;
    fp.B = B; fp.T = T; fp.K = K;
    tok_front_geometry(T, fp.SL, fp.G, fp.KW);
    if (getenv("LSD_TOKF_TRACE")) {
      // debug: phase timestamps of CTA 0 (compute warp 0: start, then [hand-over, next accumulator arrival] per phase; MMA warp:
      // [phase start, issue end]); prints after a sync, never enabled in timed runs
      static long long* dbuf = nullptr;
      if (!dbuf) cudaMalloc(&dbuf, 256 * sizeof(long long));
      cudaMemsetAsync(dbuf, 0, 256 * sizeof(long long), st);
      fp.dbg = dbuf;
      launch_tok_front(fp, st);
      std::vector<long long> hv(256);
      cudaMemcpyAsync(hv.data(), dbuf, 256 * sizeof(long long), cudaMemcpyDeviceToHost, st);
      cudaStreamSynchronize(st);
      const long long t0 = hv[128];
      fprintf(stderr, "[tokfront] compute (start=0) then (hand-over, next arrival):");
      for (int i = 0; i < 63 && hv[128 + 2 * i + 1]; ++i) fprintf(stderr, " (%lld,%lld)", hv[128 + 2 * i + 1] - t0, hv[128 + 2 * i + 2] ? hv[128 + 2 * i + 2] - t0 : 0);
      fprintf(stderr, "\n[tokfront] mma phases (start, issue-end):");
      for (int i = 0; i < 64 && hv[2 * i + 1]; ++i) fprintf(stderr, " (%lld,%lld)", hv[2 * i] - t0, hv[2 * i + 1] - t0);
      fprintf(stderr, "\n");
      fp.dbg = nullptr;
    } else
    launch_tok_front(fp, st);
    g_tl.mark(st, "T:cross");
  } else {
  fork(1);
  launch_mha_core_p(pv, 768, pa + 256, 768, pa + 512, 768, B, T, T, 8, pout(b, pbf("att1_p"), &pbf("att1_p_lo")), st);  // v2a: Q=v, K/V=a
  RUN("cross.v2a.out", a_.in = &pbf("att1_p"); a_.in_lo = &pbf("att1_p_lo"); a_.og = gt; a_.res32 = b.f("v_emb"); a_.res32_ld = 256; a_.y32 = gi; a_.y32_ld = 512;
      a_.yp = &pbf("gatein_p"); a_.yp_lo = &pbf("gatein_p_lo"));
  launch_mha_core_p(pa, 768, pv + 256, 768, pv + 512, 768, B, T, T, 8, pout(b, pbf("att2_p"), &pbf("att2_p_lo")), b1.st);  // a2v: Q=a, K/V=v
  RUNC(b1, "cross.a2v.out", a_.in = &pbf("att2_p"); a_.in_lo = &pbf("att2_p_lo"); a_.og = gt; a_.res32 = b.f("a_int"); a_.res32_ld = 256; a_.y32 = gi + 256; a_.y32_ld = 512;
      a_.yp = &pbf("gatein_p"); a_.yp_lo = &pbf("gatein_p_lo"); a_.y_plane_off = 32);
  join(1);
  RUN("cross.gate0", a_.in = &pbf("gatein_p"); a_.in_lo = &pbf("gatein_p_lo"); a_.og = gt; a_.act = ACT_GELU; a_.y32 = b.f("gate_h"); a_.y32_ld = 256);
  launch_gate_blend_p(b.f("gate_h"), b.W("cross.gate2.w"), b.W("cross.gate2.b"), gi, 512, gi + 256, 512, B * T, 256, pout(b, pbf("blend_p"), &pbf("blend_p_lo")), st);
  RUN("cross.fuse", a_.in = &pbf("blend_p"); a_.in_lo = &pbf("blend_p_lo"); a_.og = gt; a_.act = ACT_RELU; a_.y32 = b.f("fused"); a_.y32_ld = 256; a_.yp = &pbf("fused_p"); a_.yp_lo = &pbf("fused_p_lo"));
  // ---- temporal transformer (temporal.py:79-111)
  g_tl.mark(st, "T:cross");
  fork(2);
  RUNC(b1, "temporal.branch_k5", a_.in = &pbf("fused_p"); a_.in_lo = &pbf("fused_p_lo"); a_.og = gt; a_.act = ACT_GELU; a_.yp = &pbf("mscat_p"); a_.yp_lo = &pbf("mscat_p_lo"); a_.y_plane_off = 32);
  RUNC(b2, "temporal.branch_k3", a_.in = &pbf("fused_p"); a_.in_lo = &pbf("fused_p_lo"); a_.og = gt; a_.act = ACT_GELU; a_.yp = &pbf("mscat_p"); a_.yp_lo = &pbf("mscat_p_lo"); a_.y_plane_off = 0);
  launch_set_cls(b.W("temporal.cls"), tok, B, NT, 256, b2.st);
  RUN("temporal.branch_k7", a_.in = &pbf("fused_p"); a_.in_lo = &pbf("fused_p_lo"); a_.og = gt; a_.act = ACT_GELU; a_.yp = &pbf("mscat_p"); a_.yp_lo = &pbf("mscat_p_lo"); a_.y_plane_off = 64);
  join(2);
  // pre_scale_proj + residual, written straight into token rows 1..T of each window
  RUN("temporal.pre_scale_proj", a_.in = &pbf("mscat_p"); a_.in_lo = &pbf("mscat_p_lo"); a_.og = gt; a_.res32 = b.f("fused"); a_.res32_ld = 256; a_.y32 = tok; a_.y32_ld = 256;
      a_.y32_outer_stride = NT; a_.y32_row_off = 1);
  }
  // ---- the four encoder layers: one fused launch (tok_fused.cu); LSD_TOK_FUSED=0 (debug / A-B tests) or more than 64 tokens per
  // window fall back to the layer-by-layer GEMM chain
  const char* fused_env = getenv("LSD_TOK_FUSED");
  const bool fused_off = fused_env && atoi(fused_env) == 0;
  if (!fused_off && tok_fused_supported(NT)) {
    TokFusedP fp;
    memset(&fp, 0, sizeof(fp));
    fp.tok = tok;
    fp.w = reinterpret_cast<const __half*>(h->tokf_w);
    fp.stage_bytes = h->tokf_stage_bytes;
    fp.n_stage_layer = h->tokf_n_stage;
    fp.layer_bytes = h->tokf_layer_bytes;
    fp.vec = h->tokf_vec;
    fp.B = B; fp.NT = NT;
    tok_fused_geometry(NT, fp.SL, fp.G, fp.KW);
    if (getenv("LSD_TOKF_TRACE")) {
      // debug: phase timestamps of CTA 0 (MMA warp: [start, issue-end] per MMA phase; compute warp 0: [accumulator arrival,
      // hand-over] per compute phase); prints after a sync, never enabled in timed runs
      static long long* dbuf = nullptr;
      if (!dbuf) cudaMalloc(&dbuf, 384 * sizeof(long long));
      cudaMemsetAsync(dbuf, 0, 384 * sizeof(long long), st);
      fp.dbg = dbuf;
      launch_tok_fused(fp, st);
      std::vector<long long> hv(384);
      cudaMemcpyAsync(hv.data(), dbuf, 384 * sizeof(long long), cudaMemcpyDeviceToHost, st);
      cudaStreamSynchronize(st);
      const long long t0 = hv[192];
      fprintf(stderr, "[tokf] compute phases (wait-return, hand-over) cycles from start:");
      for (int i = 0; i < 96 && hv[192 + 2 * i + 1]; ++i) fprintf(stderr, " (%lld,%lld)", hv[192 + 2 * i] - t0, hv[192 + 2 * i + 1] - t0);
      fprintf(stderr, "\n[tokf] mma phases (start, issue-end):");
      for (int i = 0; i < 96 && hv[2 * i + 1]; ++i) fprintf(stderr, " (%lld,%lld)", hv[2 * i] - t0, hv[2 * i + 1] - t0);
      fprintf(stderr, "\n");
      return 0;
    }
    launch_tok_fused(fp, st);
    return 0;
  }
  const UcGeom g33 = P.g33;
  for (int l = 0; l < 4; ++l) {
    const std::string k = "t" + std::to_string(l);
    launch_layernorm_p(tok, 256, b.W((k + ".ln1.w").c_str()), b.W((k + ".ln1.b").c_str()), B * NT, 256, pout(b, pbf("tokln_p"), &pbf("tokln_p_lo")), st);
    RUN(k + ".in", a_.in = &pbf("tokln_p"); a_.in_lo = &pbf("tokln_p_lo"); a_.og = g33; a_.y32 = b.f("tok_qkv"); a_.y32_ld = 768);
    const float* qkv = b.f("tok_qkv");
    launch_mha_core_p(qkv, 768, qkv + 256, 768, qkv + 512, 768, B, NT, NT, 8, pout(b, pbf("tokatt_p"), &pbf("tokatt_p_lo")), st);
    RUN(k + ".out", a_.in = &pbf("tokatt_p"); a_.in_lo = &pbf("tokatt_p_lo"); a_.og = g33; a_.res32 = tok; a_.res32_ld = 256; a_.y32 = tok; a_.y32_ld = 256);
    launch_layernorm_p(tok, 256, b.W((k + ".ln2.w").c_str()), b.W((k + ".ln2.b").c_str()), B * NT, 256, pout(b, pbf("tokln_p"), &pbf("tokln_p_lo")), st);
    RUN(k + ".ff1", a_.in = &pbf("tokln_p"); a_.in_lo = &pbf("tokln_p_lo"); a_.og = g33; a_.act = ACT_GELU; a_.yp = &pbf("tokff_p"); a_.yp_lo = &pbf("tokff_p_lo"));
    RUN(k + ".ff2", a_.in = &pbf("tokff_p"); a_.in_lo = &pbf("tokff_p_lo"); a_.og = g33; a_.res32 = tok; a_.res32_ld = 256; a_.y32 = tok; a_.y32_ld = 256);
  }
  return 0;
}


// Zero padding of the planar buffers lives in the workspace across calls: kernels only ever write valid positions (or zeros at
// pad positions), so a workspace whose padding was initialised for these shapes is reused as is.  Three (pointer, bytes, shapes)
// signatures are remembered — slot 1 belongs to the second half of a pipelined lsd_score_windows call or to the audio groups of a
// shared-visual forward, slot 2 to the shorter last audio group of one (see VarTail), slot 0 to everything else.  A call
// invalidates every OTHER slot whose byte range overlaps this call's workspace (a forward with other shapes through the same
// memory overwrites that region's padding), and lsd_workspace_invalidate() drops all of them (the caller reused or freed the
// memory between calls).
static int ws_prepare(lsd_handle* h, const Shapes& s, const BPlan& P, char* ws, size_t ws_bytes, cudaStream_t st, int slot) {
  const int sig[6] = {s.B, s.T, s.H, s.W, s.F, s.Ta};
  WsSig& mine = h->ws_sig[slot];
  for (WsSig& other : h->ws_sig) {
    if (&other == &mine || !other.ptr) continue;
    const char* o0 = reinterpret_cast<const char*>(other.ptr);
    if (o0 < ws + ws_bytes && ws < o0 + other.bytes) other.ptr = nullptr;
  }
  if (mine.ptr == ws && mine.bytes == ws_bytes && memcmp(mine.shape, sig, sizeof(sig)) == 0) return 0;
  cudaError_t e = cudaMemsetAsync(ws + P.planar_begin, 0, P.planar_end - P.planar_begin, st);
  if (e != cudaSuccess) return lsd_fail(h, LSD_ERR_CUDA, "workspace init: %s", cudaGetErrorString(e));
  mine.ptr = ws; mine.bytes = ws_bytes; memcpy(mine.shape, sig, sizeof(sig));
  return 0;
}

// Audio side of the shared-visual forward (lsd_forward_audio_variants / lsd_score_offsets): K audio windows per video, window-major
// rows (row = b*K + k).  The visual front runs once at B; audio encoder, token path and head run at B*K in groups of gB videos
// (gB*K rows: bounded workspace, and each group's logits are one contiguous block of the (B, K) output) on a plan without video
// buffers in a workspace of their own.  A call's groups all hold gB videos except possibly the last one, which has a region of
// its own: each region keeps the zero padding of one plan shape, so repeated calls never re-zero either.
struct VarTail {
  int K = 1, gB = 1;
  char* ws = nullptr;                 // workspace of the audio plan of a full group (gB*K rows; ws_prepare slot 1) ...
  size_t ws_bytes = 0;
  char* ws_last = nullptr;            // ... and of a shorter last group (< gB*K rows; slot 2)
  size_t ws_last_bytes = 0;
  const void* audio = nullptr;        // tensor entry: (B*K, 1, F, Ta) clips of dtype adt ...
  int adt = LSD_F32;
  const float* mel_full = nullptr;    // ... or track entry: B*K mel start columns into the clip log-mel (audio == nullptr)
  int Ta_full = 0;
  const int32_t* d_astarts = nullptr;
};

static size_t dtype_bytes(int dt) { return dt == LSD_F32 ? 4 : (dt == LSD_U8 ? 1 : 2); }

// pipe_parity >= 0 (lsd_score_windows with a double workspace): everything after the visual encoder is enqueued on
// h->tail_stream, ordered after the encoder by ev_front[parity]; ev_tail_done[parity] marks the batch's logits complete.
// vt != nullptr: shared-visual forward (see VarTail); requires the fused token path (variants_shared_route) and no aux.
// feats_out (not with vt): row n receives the head's input row of window n, [cls | comb[:, 256:448]].
static int forward_bf16_impl(lsd_handle* h, const Shapes& s, float* logits, const lsd_aux* aux, char* ws, size_t ws_bytes,
                             cudaStream_t st, bool inputs_ready, const void* video, int vdt, int vlayout, const void* audio, int adt,
                             const int32_t* vstarts = nullptr, int n_frames = 0, int pipe_parity = -1, const VarTail* vt = nullptr,
                             float* feats_out = nullptr) {
  BPlan P;
  build_plan(s, P);
  if (P.f32.cursor > ws_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", P.f32.cursor, ws_bytes);
  h->stages = P.f32.stages;
  h->planar_stages.clear();
  for (const auto& kv : P.pb) {
    const PBuf& b = kv.second;
    PlanarStage ps;
    ps.off = b.off; ps.C = b.C; ps.sets = b.sets; ps.kind = b.kind; ps.map_h = b.map_h; ps.map_w = b.map_w; ps.plane_stride = b.plane_stride; ps.set_stride = b.set_stride; ps.origin = b.origin;
    ps.N = b.g.N; ps.T = b.g.T; ps.H = b.g.H; ps.W = b.g.W; ps.ot = b.g.ot; ps.oh = b.g.oh; ps.hp_extra = b.g.HP - b.g.H - b.g.oh;
    ps.ow = b.g.ow; ps.wp_extra = b.g.RW - b.g.W - b.g.ow;
    h->planar_stages[kv.first] = ps;
  }
  int rc0 = 0;
  if ((rc0 = ws_prepare(h, s, P, ws, ws_bytes, st, pipe_parity == 1 ? 1 : 0))) return rc0;
  BCtx b{h, ws, &P, st};
  const int B = s.B, T = s.T, TA = s.A4, NT = T + 1;
  auto& pb = P.pb;
  int rc = 0;
  if (!h->side_stream) {
    if (cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&h->ev_start, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_audio, cudaEventDisableTiming) != cudaSuccess)
      return lsd_fail(h, LSD_ERR_CUDA, "side stream creation failed");
  }
  cudaStream_t sst = h->side_stream;
  BCtx bs{h, ws, &P, sst};
  bs.max_ctas = h->num_sms / 2;   // measured at B=64 (re-tuned after the epilogue rewrite): 60 / 74 / 98 / 120 / 148 SMs -> 3.53 / 3.30 / 3.36 / 3.37 / 3.43 ms per step
  if (const char* e = LSD_ENV("LSD_SIDE_CTAS")) bs.max_ctas = atoi(e);   // tuning knob: SMs the side stream may occupy
  int art_ctas = bs.max_ctas;                                           // ... and during the artifact branch (tail phase)
  if (const char* e = LSD_ENV("LSD_ART_CTAS")) art_ctas = atoi(e);
  // LSD_MAIN_CTAS (tuning knob): cap the visual-encoder launches and give the audio encoder exactly the SMs they leave free
  if (const char* e = LSD_ENV("LSD_MAIN_CTAS")) { b.max_ctas = atoi(e); bs.max_ctas = h->num_sms - b.max_ctas; }
  // ---- audio encoder (independent of the video): on the side stream from the very start, so that its latency-bound chain of
  // small launches hides behind the visual encoder instead of heading the tail
  const bool audio_early = LSD_ENV("LSD_AUDIO_LATE") == nullptr;
  // Fused token path (tok_front.cu): the audio tokens' share of it — interpolation to T tokens, then ONE GEMM for
  // [a_int | cross-attention in-projection] (see pack_comb_proj in lsd_api.cu), plus a_emb itself for the aux / stage output —
  // runs right behind the audio encoder, on its stream, long before the visual encoder is done.
  const bool tcomb = token_front_enabled(T);
  auto audio_tokens = [&](const BCtx& c, const Shapes& sc) -> int {
    int rc = 0;
    const auto& q = c.P->pb;
    launch_lerp_tokens_p(c.f("a_feat"), c.f("a_fint"), sc.B, sc.A4, sc.T, 256, pout(c, q.at("afint_p"), &q.at("afint_p_lo")), c.st);
    RUNC(c, "cross.acomb", a_.in = &q.at("afint_p"); a_.in_lo = &q.at("afint_p_lo"); a_.og = c.P->gt; a_.y32 = c.f("acomb"); a_.y32_ld = 1024);
    // a_emb itself (TA tokens per window) is an aux output only: the token path consumes the interpolated rows above
    if (aux && aux->audio_tokens) RUNC(c, "projection.audio_proj", a_.in = &q.at("afeat_p"); a_.in_lo = &q.at("afeat_p_lo"); a_.og = c.P->gta; a_.y32 = c.f("a_emb"); a_.y32_ld = 256);
    return 0;
  };
  // shared-visual forward: plans of the audio groups (the last group may hold fewer videos) and the audio side of group g
  const int n_groups = vt ? (B + vt->gB - 1) / vt->gB : 0;
  const bool short_last = vt && B - (n_groups - 1) * vt->gB < vt->gB;   // the last group holds fewer than gB videos
  auto plan_of = [&](int g) { return short_last && g == n_groups - 1 ? 1 : 0; };
  Shapes sA[2];
  BPlan PA[2];
  char* aws[2] = {nullptr, nullptr};
  if (vt) {
    aws[0] = vt->ws; aws[1] = vt->ws_last;
    for (int i = 0; i < 2; ++i) {
      if (i != plan_of(0) && i != plan_of(n_groups - 1)) continue;
      const int nb = i == 0 ? vt->gB : B - (n_groups - 1) * vt->gB;
      const size_t cap = i == 0 ? vt->ws_bytes : vt->ws_last_bytes;
      if ((rc = make_shapes(h, nb * vt->K, T, 16, 16, s.F, s.Ta, sA[i]))) return rc;
      build_plan(sA[i], PA[i], false);
      if (!aws[i] || PA[i].f32.cursor > cap) return lsd_fail(h, LSD_ERR_WORKSPACE, "audio-variant workspace too small: need %zu bytes, got %zu", PA[i].f32.cursor, cap);
    }
  }
  auto var_audio = [&](int g, cudaStream_t stream, int max_ctas) -> int {
    const int pi = plan_of(g);
    int rc = ws_prepare(h, sA[pi], PA[pi], aws[pi], pi ? vt->ws_last_bytes : vt->ws_bytes, stream, 1 + pi);
    if (rc) return rc;
    BCtx c{h, aws[pi], &PA[pi], stream};
    c.max_ctas = max_ctas;
    const size_t r0 = (size_t)g * vt->gB * vt->K;
    if (vt->d_astarts) launch_gather_audio(vt->mel_full, s.F, vt->Ta_full, vt->d_astarts + r0, c.f("aud"), sA[pi].B, s.Ta, stream);
    const void* au = vt->audio ? reinterpret_cast<const char*>(vt->audio) + r0 * s.F * s.Ta * dtype_bytes(vt->adt) : nullptr;
    if ((rc = audio_encoder_bf16(c, sA[pi], vt->d_astarts != nullptr, au, vt->adt))) return rc;
    return audio_tokens(c, sA[pi]);
  };
  g_tl.on = LSD_ENV("LSD_TIMELINE") != nullptr;
  g_tl.mark(st, "start");
  if (vt) {                             // the first audio group takes the audio encoder's place next to the visual encoder
    cudaEventRecord(h->ev_start, st);
    cudaStreamWaitEvent(sst, h->ev_start, 0);
    if ((rc = var_audio(0, sst, bs.max_ctas))) return rc;
    cudaEventRecord(h->ev_audio, sst);
  } else if (audio_early) {
    cudaEventRecord(h->ev_start, st);
    cudaStreamWaitEvent(sst, h->ev_start, 0);
    if ((rc = audio_encoder_bf16(bs, s, inputs_ready, audio, adt))) return rc;
    if (tcomb && (rc = audio_tokens(bs, s))) return rc;
    g_tl.mark(sst, "S:audio_enc");
    cudaEventRecord(h->ev_audio, sst);
  }
  // ---- video -> bf16 pixel rows (+ per-frame laplacian conv), stem conv on tcgen05 (Toeplitz K), max-pool in planar layout
  const PBuf &xs = pb["xs"], &xl = pb["xl"], &so = pb["s_out"], &x1 = pb["x1"];
  const float* lapw = h->warena + h->convs.at("art.lap").w_off;
  // (vstarts: the uint8 track is read in place, window n = frames vstarts[n] .. vstarts[n]+T-1 — no fp32 window copy)
  if (vstarts) launch_video_rows(video, vdt, vlayout, lapw, h->lapw_host, b.org(xs), b.org(xl), xs.set_stride, xs.g, s.H, s.W, st, h->num_sms, vstarts, n_frames);
  else if (inputs_ready) launch_video_rows(b.f("vid"), LSD_F32, LSD_NDHWC, lapw, h->lapw_host, b.org(xs), b.org(xl), xs.set_stride, xs.g, s.H, s.W, st, h->num_sms);
  else launch_video_rows(video, vdt, vlayout, lapw, h->lapw_host, b.org(xs), b.org(xl), xs.set_stride, xs.g, s.H, s.W, st, h->num_sms);
  g_tl.mark(st, "M:video_rows");
  float* comb = b.f("comb");
  PlanarOut none{nullptr, nullptr, 0, 0, 0, 0};
  const PBuf& hf = pb["hf_f"];
  // Stem + max-pool.  Default: the temporal-ring kernel (stem_ring.cu: the three temporal taps as one N = 192 MMA); LSD_STEM_RING=0,
  // rows too wide for the ring or non-canonical stem weights take the flat shift-GEMM launch (CTA pairs).  The summation order
  // differs between the two, the bits of a given route do not depend on the batch.
  static const bool ring_env = !(LSD_ENV("LSD_STEM_RING") && atoi(LSD_ENV("LSD_STEM_RING")) == 0);
  if (ring_env && h->stem_ring_w_off != 0 && 128 + 3 * xs.g.RW + 3 <= 640) {
    if ((rc = run_stem_ring(b, xs, so))) return rc;
  } else {
    RUN("visual_encoder.stem", a_.in = &xs; a_.og = xs.g; a_.act = ACT_RELU; a_.yp = &so);
  }
  g_tl.mark(st, "M:stem");
  launch_planar_maxpool(b.org(so), so.plane_stride, so.g, b.org(x1), x1.plane_stride, x1.g, 64, st);
  g_tl.mark(st, "M:maxpool");
  // ---- residual stages (visual_encoder.py:81-87, 133-152)
  if ((rc = res_stage_umma(b, "visual_encoder.layer1", x1, pb["l1a"], pb["y1"], false, UC_Y_PARITY))) return rc;
  g_tl.mark(st, "M:layer1");
  // layer2 writes y2 folded when layer3 runs on the folded route (small maps, see fold_route); y4 is always the plain padded map
  if ((rc = res_stage_umma(b, "visual_encoder.layer2", pb["y1"], pb["l2a"], pb["y2"], true, P.fold3 ? UC_Y_FOLD : UC_Y_PARITY))) return rc;
  g_tl.mark(st, "M:layer2");
  if (P.fold3) rc = res_stage_fold(b, "visual_encoder.layer3", pb["y2"], s.H2, s.W2, pb["l3a"], s.H3, s.W3, pb["y3"], UC_Y_FOLD);
  else rc = res_stage_umma(b, "visual_encoder.layer3", pb["y2"], pb["l3a"], pb["y3"], true, P.fold4 ? UC_Y_FOLD : UC_Y_PARITY);
  if (rc) return rc;
  g_tl.mark(st, "M:layer3");
  if (P.fold4) rc = res_stage_fold(b, "visual_encoder.layer4", pb["y3"], s.H3, s.W3, pb["l4a"], s.H4, s.W4, pb["y4"], UC_Y_MAP);
  else rc = res_stage_umma(b, "visual_encoder.layer4", pb["y3"], pb["l4a"], pb["y4"], true, UC_Y_PLAIN);
  if (rc) return rc;
  g_tl.mark(st, "M:layer4");
  b.max_ctas = 0;
  const PBuf& y4 = pb["y4"];
  // spatial mean -> visual tokens (fp32 stage + planar GEMM input)
  launch_planar_mean2(b.org(y4), y4.plane_stride, y4.g, 256, b.f("v_feat"), 256, 0, pout(b, pb["vfeat_p"], &pb["vfeat_p_lo"]), st);
  // ---- artifact detector (artifact_detector.py:149-183) on a side stream: its convolutions (hf front/back on the laplacian
  // rows, temporal-inconsistency convs on the feature map and on its temporal delta) only need the visual encoder's
  // output, so they run concurrently with the audio encoder + token path, whose small grids leave most SMs idle.
  cudaEventRecord(h->ev_fork, st);
  cudaStreamWaitEvent(sst, h->ev_fork, 0);
  const bool skip_art = LSD_ENV("LSD_SKIP_ART") != nullptr;   // timing experiment only (garbage logits)
  bs.max_ctas = art_ctas;
  if (!skip_art) {
  RUNS("art.td0", a_.in = &y4; a_.og = y4.g; a_.act = ACT_RELU; a_.yp = &pb["art_a"]);
  RUNS("art.td3", a_.in = &pb["art_a"]; a_.og = y4.g; a_.act = ACT_RELU; a_.yp = &pb["art_b"]);
  launch_planar_mean2(bs.org(pb["art_b"]), pb["art_b"].plane_stride, y4.g, 64, comb + 256, 448, 1, none, sst);
  g_tl.mark(sst, "S:td_feat");
  const PBuf& dl = pb["delta"];
  if (T > 1) launch_planar_delta(bs.org(y4), y4.plane_stride, y4.g, bs.org(dl), dl.plane_stride, dl.g, 256, sst);
  // (T == 1: the delta map is all zeros — the buffer is never written and keeps its zero initialisation)
  RUNS("art.td0", a_.in = &dl; a_.og = dl.g; a_.act = ACT_RELU; a_.yp = &pb["artd_a"]);
  RUNS("art.td3", a_.in = &pb["artd_a"]; a_.og = dl.g; a_.act = ACT_RELU; a_.yp = &pb["artd_b"]);
  launch_planar_mean2(bs.org(pb["artd_b"]), pb["artd_b"].plane_stride, dl.g, 64, comb + 320, 448, 1, none, sst);
  g_tl.mark(sst, "S:td_delta");
  // high-frequency branch: Conv3d 3->32 s(1,2,2) on the laplacian pixel rows (Toeplitz K), Conv3d 32->64 s(1,2,2) planar.
  // It depends on nothing but the laplacian rows, so in the tail it runs on a second side stream NEXT TO the
  // temporal-inconsistency convolutions instead of behind them: both chains are capped at half of the SMs, and the token path's
  // small grids fit in between (also when batches are pipelined: 10k-window run 19.6k -> 20.5k windows/s).
  if (!h->side2_stream) {
    if (cudaStreamCreateWithFlags(&h->side2_stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&h->ev_join2, cudaEventDisableTiming) != cudaSuccess)
      return lsd_fail(h, LSD_ERR_CUDA, "second side stream creation failed");
  }
  const cudaStream_t hst = h->side2_stream;
  cudaStreamWaitEvent(hst, h->ev_fork, 0);
  BCtx bh = bs;
  bh.st = hst;
  if (const char* e = LSD_ENV("LSD_HF_CTAS")) bh.max_ctas = atoi(e);
  RUNC(bh, "art.hf0", a_.in = &xl; a_.og = xl.g; a_.act = ACT_RELU; a_.yp = &hf);
  g_tl.mark(hst, "S:hf0");
  RUNC(bh, "art.hf3", a_.in = &hf; a_.og = hf.g; a_.act = ACT_RELU; a_.yp = &pb["hf_b"]);
  launch_planar_mean2(bh.org(pb["hf_b"]), pb["hf_b"].plane_stride, hf.g, 64, comb + 384, 448, 1, none, hst);
  g_tl.mark(hst, "S:hf3");
  // fold the second side stream back into the first: ev_join then covers both
  cudaEventRecord(h->ev_join2, hst);
  cudaStreamWaitEvent(sst, h->ev_join2, 0);
  }
  cudaEventRecord(h->ev_join, sst);
  // ---- everything below is the latency-bound tail (small grids): on the caller's stream, or on the tail stream when batches
  // are pipelined (the main stream then goes straight on to the next batch's visual encoder)
  cudaStream_t tst = st;
  if (pipe_parity >= 0) {
    cudaEventRecord(h->ev_front[pipe_parity], st);
    cudaStreamWaitEvent(h->tail_stream, h->ev_front[pipe_parity], 0);
    tst = h->tail_stream;
  }
  {
  BCtx b{h, ws, &P, tst};
  cudaStream_t st = tst;
  HeadW hw;
  auto cw = [&](const char* key) { return h->warena + h->convs.at(key).w_off; };
  auto cb = [&](const char* key) { return h->warena + h->convs.at(key).shift_off; };
  hw.w0 = cw("art.fuse0"); hw.b0 = cb("art.fuse0"); hw.w2 = cw("art.fuse2"); hw.b2 = cb("art.fuse2");
  hw.wc = cw("head.fc0"); hw.bc = cb("head.fc0");
  hw.lng = b.W("head.ln.w"); hw.lnb = b.W("head.ln.b"); hw.wo = b.W("head.out.w"); hw.bo = b.W("head.out.b");
  if (vt) {
    // token path + head per audio group: row b*K + k reads the visual projection and artifact features of video b
    RUN("cross.vcomb", a_.in = &pb["vfeat_p"]; a_.in_lo = &pb["vfeat_p_lo"]; a_.og = P.gt; a_.y32 = b.f("vcomb"); a_.y32_ld = 1024);
    for (int g = 0; g < n_groups; ++g) {
      if (g == 0) cudaStreamWaitEvent(st, h->ev_audio, 0);
      else if ((rc = var_audio(g, st, 0))) return rc;       // (the previous group's token path and head are done with this workspace)
      const int pi = plan_of(g), b0 = g * vt->gB;
      BCtx c{h, aws[pi], &PA[pi], st};
      if ((rc = token_path_bf16(c, sA[pi], true, b.f("vcomb") + (size_t)b0 * T * 1024, vt->K))) return rc;
      if (g == 0) cudaStreamWaitEvent(st, h->ev_join, 0);   // artifact features (comb[:, 256:448]) are complete
      launch_head(c.f("tok"), (int64_t)NT * 256, comb + (size_t)b0 * 448, hw, logits + (size_t)b0 * vt->K, sA[pi].B, st, vt->K);
    }
    if (pipe_parity >= 0) cudaEventRecord(h->ev_tail_done[pipe_parity], st);
    return 0;
  }
  if (!audio_early) { if ((rc = audio_encoder_bf16(b, s, inputs_ready, audio, adt))) return rc; }
  // ---- projection (fusion_module.py:108-124)
  const UcGeom gt = P.gt;
  if (tcomb) {
    // fused token path: one GEMM gives [v_emb | cross-attention in-projection] per visual token (the audio half ran behind the audio encoder)
    if (!audio_early) { if ((rc = audio_tokens(b, s))) return rc; }
    RUN("cross.vcomb", a_.in = &pb["vfeat_p"]; a_.in_lo = &pb["vfeat_p_lo"]; a_.og = gt; a_.y32 = b.f("vcomb"); a_.y32_ld = 1024);
    if (audio_early) cudaStreamWaitEvent(st, h->ev_audio, 0);   // [a_int | in-projection] of the audio tokens is complete
  } else {
    RUN("projection.visual_proj", a_.in = &pb["vfeat_p"]; a_.in_lo = &pb["vfeat_p_lo"]; a_.og = gt; a_.yp = &pb["vemb_p"]; a_.yp_lo = &pb["vemb_p_lo"]; a_.y32 = b.f("v_emb"); a_.y32_ld = 256);
    if (audio_early) cudaStreamWaitEvent(st, h->ev_audio, 0);   // audio features (a_feat / afeat_p) are complete
    RUN("projection.audio_proj", a_.in = &pb["afeat_p"]; a_.in_lo = &pb["afeat_p_lo"]; a_.og = P.gta; a_.y32 = b.f("a_emb"); a_.y32_ld = 256);
  }
  g_tl.mark(st, "T:proj");
  if ((rc = token_path_bf16(b, s, tcomb))) return rc;
  float* tok = b.f("tok");
  g_tl.mark(st, "T:tokens");
  // cls = tok[:,0]: no final norm (temporal.py:110-111); the head reads the CLS rows in place
  cudaStreamWaitEvent(st, h->ev_join, 0);   // artifact features (comb[:, 256:448]) are complete
  // ---- artifact fusion MLP + classification head, fused, fp32 (artifact_detector.py:142-147,180-181; classifier.py:14-34)
  launch_head(tok, (int64_t)NT * 256, comb, hw, logits, B, st);
  if (feats_out) {   // on the head's stream, before ev_tail_done: the pipelined tails reuse this workspace half afterwards
    launch_copy_rows(tok, (int64_t)NT * 256, feats_out, LSD_BRANCH_FEATURES, B, 256, st);
    launch_copy_rows(comb + 256, 448, feats_out + 256, LSD_BRANCH_FEATURES, B, 192, st);
  }
  g_tl.mark(st, "T:head");
  g_tl.dump();
  if (aux) {
    const size_t tb = (size_t)B * T * 256 * sizeof(float);
    if (aux->visual_tokens) {
      if (tcomb) launch_copy_rows(b.f("vcomb"), 1024, aux->visual_tokens, 256, B * T, 256, st);   // v_emb = the first 256 columns of the merged projection
      else cudaMemcpyAsync(aux->visual_tokens, b.f("v_emb"), tb, cudaMemcpyDeviceToDevice, st);
    }
    if (aux->audio_tokens) cudaMemcpyAsync(aux->audio_tokens, b.f("a_emb"), (size_t)B * TA * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (aux->fused_tokens) cudaMemcpyAsync(aux->fused_tokens, b.f("fused"), tb, cudaMemcpyDeviceToDevice, st);
    if (aux->cls_output) launch_copy_rows(tok, (int64_t)NT * 256, aux->cls_output, 256, B, 256, st);
  }
  if (pipe_parity >= 0) cudaEventRecord(h->ev_tail_done[pipe_parity], st);
  }
  return 0;
}

// Introspection (tests): a planar bf16 buffer of the last tensor-core forward -> fp32 channels-last (N, T, Hf, Wf, C).
// (Hf, Wf) must be the full-resolution extent of the map the buffer holds (recorded by build_plan), whatever its layout: the unpack
// kernel derives its addressing from (sets, Hf, Wf), so any other extent would read outside the buffer.  name_lo: optional low
// part of a (hi, lo) pair, added in; it must have the layout of the high part.
int planar_stage_read(lsd_handle* h, const char* name, const char* name_lo, const char* ws, float* out, int64_t out_elems, int Hf, int Wf,
                      cudaStream_t st) {
  auto it = h->planar_stages.find(name);
  if (it == h->planar_stages.end()) return lsd_fail(h, LSD_ERR_ARG, "unknown planar stage %s", name);
  const PlanarStage& ps = it->second;
  const PlanarStage* pl = nullptr;
  if (name_lo && *name_lo) {
    auto il = h->planar_stages.find(name_lo);
    if (il == h->planar_stages.end()) return lsd_fail(h, LSD_ERR_ARG, "unknown planar stage %s", name_lo);
    pl = &il->second;
  }
  if (ps.kind == PK_ROWS) return lsd_fail(h, LSD_ERR_ARG, "stage %s holds pixel rows, not a channel map", name);
  if (Hf != ps.map_h || Wf != ps.map_w)
    return lsd_fail(h, LSD_ERR_SHAPE, "stage %s holds a %d x %d map, got %d x %d", name, ps.map_h, ps.map_w, Hf, Wf);
  if (pl && (pl->kind != ps.kind || pl->C != ps.C || pl->sets != ps.sets || pl->map_h != ps.map_h || pl->map_w != ps.map_w ||
             pl->plane_stride != ps.plane_stride || pl->set_stride != ps.set_stride || pl->origin != ps.origin || pl->N != ps.N ||
             pl->T != ps.T || pl->H != ps.H || pl->W != ps.W || pl->ot != ps.ot || pl->oh != ps.oh || pl->hp_extra != ps.hp_extra ||
             pl->ow != ps.ow || pl->wp_extra != ps.wp_extra))
    return lsd_fail(h, LSD_ERR_SHAPE, "stage %s does not have the layout of %s", name_lo, name);
  const UcGeom g = make_geom_ex(ps.N, ps.T, ps.H, ps.W, ps.ot, ps.oh, ps.hp_extra, ps.ow, ps.wp_extra);
  // the layout unpack_planar_any_kernel selects for the true extent must be the recorded one (a folded 1 x 1 map is plain, and the
  // two parity splits address a 1-wide map alike)
  const int sel = ps.sets == 1 ? PK_PLAIN : (g.SL == 1 && ps.sets == Hf * Wf) ? PK_FOLD : Wf == g.W ? PK_PARITY_H : PK_PARITY_HW;
  const int want = (ps.kind == PK_FOLD && ps.sets == 1) ? PK_PLAIN : (ps.kind == PK_PARITY_HW && Wf == 1) ? PK_PARITY_H : ps.kind;
  if (sel != want) return lsd_fail(h, LSD_ERR_SHAPE, "stage %s: layout %d cannot be unpacked (reads as %d)", name, ps.kind, sel);
  if ((int64_t)ps.N * ps.T * Hf * Wf * ps.C != out_elems) return lsd_fail(h, LSD_ERR_SHAPE, "stage %s holds %lld elements", name, (long long)ps.N * ps.T * Hf * Wf * ps.C);
  const __nv_bfloat16* x = reinterpret_cast<const __nv_bfloat16*>(ws + ps.off) + ps.origin;
  const __nv_bfloat16* xlo = pl ? reinterpret_cast<const __nv_bfloat16*>(ws + pl->off) + pl->origin : nullptr;
  launch_unpack_planar_any(x, xlo, ps.plane_stride, ps.set_stride, g, ps.C, ps.sets, Hf, Wf, out, st);
  return 0;
}

int ensure_pipeline(lsd_handle* h) {
  if (h->tail_stream) return 0;
  if (cudaStreamCreateWithFlags(&h->tail_stream, cudaStreamNonBlocking) != cudaSuccess) return lsd_fail(h, LSD_ERR_CUDA, "tail stream creation failed");
  for (int i = 0; i < 2; ++i)
    if (cudaEventCreateWithFlags(&h->ev_front[i], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_tail_done[i], cudaEventDisableTiming) != cudaSuccess)
      return lsd_fail(h, LSD_ERR_CUDA, "pipeline event creation failed");
  return 0;
}

// ---- sub-paths behind the C-ABI (lsd_audio_encoder / lsd_token_path): the same functions the full forward runs, on a plan
// whose unused video extents are minimal (16x16, one frame), so the audits of BASELINE.json configs 3 and 4 can sweep the batch.
static int subpath_begin(lsd_handle* h, const Shapes& s, BPlan& P, char* ws, size_t ws_bytes, cudaStream_t st) {
  build_plan(s, P);
  if (P.f32.cursor > ws_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", P.f32.cursor, ws_bytes);
  h->stages = P.f32.stages;
  if (int rc = ws_prepare(h, s, P, ws, ws_bytes, st, 0)) return rc;
  return 0;
}

size_t audio_encoder_bf16_bytes(lsd_handle* h, int B, int F, int Ta) {
  Shapes s;
  if (make_shapes(h, B, 1, 16, 16, F, Ta, s) != 0) return 0;
  BPlan P;
  build_plan(s, P);
  return P.f32.cursor + 256;
}

int audio_encoder_bf16_run(lsd_handle* h, int B, int F, int Ta, const void* audio, int adt, float* feats_out, char* ws, size_t ws_bytes,
                           cudaStream_t st) {
  Shapes s;
  int rc = make_shapes(h, B, 1, 16, 16, F, Ta, s);
  if (rc) return rc;
  BPlan P;
  if ((rc = subpath_begin(h, s, P, ws, ws_bytes, st))) return rc;
  BCtx b{h, ws, &P, st};
  if ((rc = audio_encoder_bf16(b, s, false, audio, adt))) return rc;
  cudaMemcpyAsync(feats_out, b.f("a_feat"), (size_t)B * s.A4 * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st);
  return 0;
}

size_t token_path_bf16_bytes(lsd_handle* h, int B, int T, int TA) {
  Shapes s;
  if (make_shapes(h, B, T, 16, 16, 16, 8 * TA, s) != 0) return 0;
  BPlan P;
  build_plan(s, P);
  return P.f32.cursor + 256;
}

int token_path_bf16_run(lsd_handle* h, int B, int T, int TA, const float* v_emb, const float* a_emb, float* fused_out, float* cls_out,
                        char* ws, size_t ws_bytes, cudaStream_t st) {
  Shapes s;
  int rc = make_shapes(h, B, T, 16, 16, 16, 8 * TA, s);
  if (rc) return rc;
  if (s.A4 != TA) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_token_path: unsupported audio token count %d", TA);
  BPlan P;
  if ((rc = subpath_begin(h, s, P, ws, ws_bytes, st))) return rc;
  BCtx b{h, ws, &P, st};
  // projected embeddings arrive as fp32 rows; the planar (hi, lo) copy of v_emb is what projection.visual_proj's epilogue writes
  cudaMemcpyAsync(b.f("a_emb"), a_emb, (size_t)B * TA * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st);
  launch_lerp_tokens_p(v_emb, b.f("v_emb"), B, T, T, 256, pout(b, P.pb.at("vemb_p"), &P.pb.at("vemb_p_lo")), st);
  if ((rc = token_path_bf16(b, s))) return rc;
  if (fused_out) cudaMemcpyAsync(fused_out, b.f("fused"), (size_t)B * T * 256 * sizeof(float), cudaMemcpyDeviceToDevice, st);
  if (cls_out) launch_copy_rows(b.f("tok"), (int64_t)(T + 1) * 256, cls_out, 256, B, 256, st);
  return 0;
}

int forward_bf16(lsd_handle* h, int B, int T, int H, int W, int F, int Ta, const void* video, int vdt, int vlayout,
                 const void* audio, int adt, float* logits, const lsd_aux* aux, char* ws, size_t ws_bytes, cudaStream_t st,
                 bool inputs_ready) {
  Shapes s;
  int rc = make_shapes(h, B, T, H, W, F, Ta, s);
  if (rc) return rc;
  return forward_bf16_impl(h, s, logits, aux, ws, ws_bytes, st, inputs_ready, video, vdt, vlayout, audio, adt);
}

int score_batch_bf16(lsd_handle* h, const uint8_t* track, int n_frames, const int32_t* d_vstarts, const int32_t* d_astarts,
                     const float* mel_full, int Ta_full, int nb, int T, int H, int W, int F, int Ta, float* logits, char* ws,
                     size_t ws_bytes, cudaStream_t st, int pipe_parity, float* feats_out) {
  Shapes s;
  int rc = make_shapes(h, nb, T, H, W, F, Ta, s);
  if (rc) return rc;
  BPlan P;
  build_plan(s, P);
  if (P.f32.cursor > ws_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", P.f32.cursor, ws_bytes);
  BCtx b{h, ws, &P, st};
  launch_gather_audio(mel_full, F, Ta_full, d_astarts, b.f("aud"), nb, Ta, st);
  if (video_rows_bulk_ok(track, LSD_U8, LSD_NDHWC, W))
    return forward_bf16_impl(h, s, logits, nullptr, ws, ws_bytes, st, true, track, LSD_U8, LSD_NDHWC, nullptr, 0, d_vstarts, n_frames, pipe_parity,
                             nullptr, feats_out);
  launch_gather_windows_u8(track, n_frames, d_vstarts, b.f("vid"), nb, T, H * W * 3, st);
  return forward_bf16_impl(h, s, logits, nullptr, ws, ws_bytes, st, true, nullptr, 0, 0, nullptr, 0, nullptr, 0, pipe_parity, nullptr, feats_out);
}

// ---- shared-visual forward (lsd_forward_audio_variants / lsd_score_offsets)
// The route needs the fused token kernels (tok_front reads the visual rows of its window group); every other configuration
// scores one plain forward per audio variant instead (lsd_api.cu).
bool variants_shared_route(int T) {
  const char* fe = getenv("LSD_TOK_FUSED");
  return token_front_enabled(T) && !(fe && atoi(fe) == 0) && tok_fused_supported(T + 1);
}

// Videos per audio group: at most LSD_VARIANT_ROWS (default 512) rows of B*K run through the audio side at once.  A group holds
// whole videos, so its logits are a contiguous block of the (B, K) output; results do not depend on the grouping.
static int variants_group(int B, int K) {
  int cap = 512;
  if (const char* e = getenv("LSD_VARIANT_ROWS")) cap = std::max(1, atoi(e));
  const int per = std::max(1, cap / K);
  const int n_groups = (B + per - 1) / per;
  return std::max(1, (B + n_groups - 1) / n_groups);   // equal groups where B allows it: one audio plan for every group
}

static size_t variants_visual_bytes(const Shapes& s) {
  BPlan P;
  build_plan(s, P);
  return (P.f32.cursor + 255) & ~size_t(255);
}

// audio plan of `rows` rows (see VarTail), 256-byte aligned; 0 for rows < 1
static size_t variants_audio_bytes(int rows, int T, int F, int Ta) {
  Shapes sa;
  if (rows < 1 || make_shapes(nullptr, rows, T, 16, 16, F, Ta, sa) != 0) return 0;
  BPlan PA;
  build_plan(sa, PA, false);
  return (PA.f32.cursor + 255) & ~size_t(255);
}

// Every call with at most `B` videos fits: the groups are sized from B (variants_group), a call with fewer videos keeps that
// group size, and its shorter last group (at most gB - 1 videos) has its own region.
size_t variants_bf16_bytes(lsd_handle* h, int B, int K, int T, int H, int W, int F, int Ta) {
  Shapes s;
  if (B < 1 || K < 1 || make_shapes(h, B, T, H, W, F, Ta, s) != 0) return 0;
  const int gB = variants_group(B, K);
  const size_t a0 = variants_audio_bytes(gB * K, T, F, Ta);
  if (a0 == 0) return 0;
  return variants_visual_bytes(s) + a0 + variants_audio_bytes((gB - 1) * K, T, F, Ta) + 256;
}

// ws: [visual plan at nb videos | audio plan of a full group | audio plan of a shorter last group].  plan_B: the largest call the
// workspace was sized for (variants_bf16_bytes); the group size follows it, not nb, so a short last batch stays within the sizing.
static int variants_run(lsd_handle* h, const Shapes& s, int plan_B, VarTail& vt, float* logits, char* ws, size_t ws_bytes, cudaStream_t st,
                        bool inputs_ready, const void* video, int vdt, int vlayout, const int32_t* vstarts, int n_frames) {
  const size_t vb = variants_visual_bytes(s);
  vt.gB = variants_group(plan_B, vt.K);
  const size_t a0 = variants_audio_bytes(vt.gB * vt.K, s.T, s.F, s.Ta);
  if (vb + a0 > ws_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need more than %zu bytes, got %zu", vb + a0, ws_bytes);
  vt.ws = ws + vb;
  vt.ws_bytes = a0;
  vt.ws_last = ws + vb + a0;
  vt.ws_last_bytes = ws_bytes - vb - a0;
  return forward_bf16_impl(h, s, logits, nullptr, ws, vb, st, inputs_ready, video, vdt, vlayout, nullptr, 0, vstarts, n_frames, -1, &vt);
}

int forward_variants_bf16(lsd_handle* h, int B, int K, int T, int H, int W, int F, int Ta, const void* video, int vdt, int vlayout,
                          const void* audio, int adt, float* logits, char* ws, size_t ws_bytes, cudaStream_t st) {
  Shapes s;
  int rc = make_shapes(h, B, T, H, W, F, Ta, s);
  if (rc) return rc;
  VarTail vt;
  vt.K = K; vt.audio = audio; vt.adt = adt;
  return variants_run(h, s, B, vt, logits, ws, ws_bytes, st, false, video, vdt, vlayout, nullptr, 0);
}

int score_offsets_batch_bf16(lsd_handle* h, const uint8_t* track, int n_frames, const int32_t* d_vstarts, const int32_t* d_astarts,
                             const float* mel_full, int Ta_full, int nb, int batch, int K, int T, int H, int W, int F, int Ta, float* logits,
                             char* ws, size_t ws_bytes, cudaStream_t st) {
  Shapes s;
  int rc = make_shapes(h, nb, T, H, W, F, Ta, s);
  if (rc) return rc;
  VarTail vt;
  vt.K = K; vt.mel_full = mel_full; vt.Ta_full = Ta_full; vt.d_astarts = d_astarts;
  if (video_rows_bulk_ok(track, LSD_U8, LSD_NDHWC, W))
    return variants_run(h, s, batch, vt, logits, ws, ws_bytes, st, true, track, LSD_U8, LSD_NDHWC, d_vstarts, n_frames);
  BPlan P;
  build_plan(s, P);
  BCtx b{h, ws, &P, st};
  launch_gather_windows_u8(track, n_frames, d_vstarts, b.f("vid"), nb, T, H * W * 3, st);
  return variants_run(h, s, batch, vt, logits, ws, ws_bytes, st, true, nullptr, 0, 0, nullptr, 0);
}
