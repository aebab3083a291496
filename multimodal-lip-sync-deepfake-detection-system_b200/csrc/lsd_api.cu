// C-ABI of liblsd_b200.so (include/lsd_b200.h): handle, weight packing (BN fold), forward orchestration.
// Host-side only; every numeric op is a kernel from kernels_f32.cu / logmel.cu / umma_conv.cu.
#include "../../include/lsd_b200.h"
#include "lsd_kernels.h"
#include "lsd_internal.h"

#include <algorithm>
#include <cmath>
#include <initializer_list>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>

#include "forward_common.h"
#include "tok_front.cuh"
#include "tok_fused.cuh"
#include "stem_ring.cuh"
#include "umma_conv.cuh"
#include "token_kernels.cuh"
using namespace lsd;

static thread_local std::string g_create_error;

int lsd_fail(lsd_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

#define CUDA_OK(h, expr)                                                                              \
  do {                                                                                                \
    cudaError_t e_ = (expr);                                                                          \
    if (e_ != cudaSuccess) return lsd_fail(h, LSD_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
  } while (0)

// Every entry point makes the handle's device current for its own work and restores the caller's device on return
// (torch reads the current device from the runtime: switching it behind the caller's back would misplace later allocations).
namespace {
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) err = cudaSetDevice(dev);
    else prev = -1;   // nothing to restore
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
}  // namespace
#define ENTER_DEVICE(h)                 \
  DeviceGuard dev_guard_((h)->device);  \
  CUDA_OK(h, dev_guard_.err)

extern "C" int lsd_version(void) { return 200; }

extern "C" const char* lsd_last_error(lsd_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

extern "C" int lsd_create(lsd_handle** out, int device) {
  if (!out) return lsd_fail(nullptr, LSD_ERR_ARG, "lsd_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return lsd_fail(nullptr, LSD_ERR_CUDA, "lsd_create: no CUDA device (%s); this library has no CPU fallback",
                    cudaGetErrorString(e));
  if (device < 0 || device >= count) return lsd_fail(nullptr, LSD_ERR_ARG, "lsd_create: bad device %d", device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return lsd_fail(nullptr, LSD_ERR_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10)
    return lsd_fail(nullptr, LSD_ERR_UNSUPPORTED, "lsd_create: device %d is sm_%d%d; this library is built for sm_100a only",
                    device, prop.major, prop.minor);
  lsd_handle* h = new lsd_handle();
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  h->launches0 = kernel_launches();
  DeviceGuard guard(device);
  if (guard.err != cudaSuccess) { delete h; return lsd_fail(nullptr, LSD_ERR_CUDA, "lsd_create: cudaSetDevice(%d): %s", device, cudaGetErrorString(guard.err)); }
  // per-device state (opt-in shared-memory limits, __constant__ twiddles) is set up for every handle: cheap, and correct
  // when one process holds handles on several devices
  int rc = init_logmel_tables(h);
  if (rc == 0) {
    cudaError_t ce = lsd::umma_conv_device_init();
    if (ce == cudaSuccess) ce = lsd::tok_fused_device_init();
    if (ce == cudaSuccess) ce = lsd::stem_ring_device_init();
    if (ce == cudaSuccess) ce = lsd::tok_front_device_init();
    if (ce == cudaSuccess) ce = lsd::warp_windows_device_init();
    if (ce == cudaSuccess) ce = lsd::jpeg_windows_device_init();
    if (ce == cudaSuccess) ce = lsd::resize_windows_device_init();
    if (ce == cudaSuccess) ce = lsd::attribution_device_init();
    if (ce != cudaSuccess) rc = lsd_fail(h, LSD_ERR_CUDA, "lsd_create: kernel attribute setup: %s", cudaGetErrorString(ce));
  }
  if (rc != 0) { g_create_error = h->err; delete h; return rc; }
  *out = h;
  return LSD_OK;
}

extern "C" void lsd_destroy(lsd_handle* h) {
  if (!h) return;
  DeviceGuard guard(h->device);
  if (h->warena) cudaFree(h->warena);
  if (h->barena) cudaFree(h->barena);
  if (h->bbias) cudaFree(h->bbias);
  if (h->tokfr_w) cudaFree(h->tokfr_w);
  if (h->tokfr_vec) cudaFree(h->tokfr_vec);
  if (h->tokf_w) cudaFree(h->tokf_w);
  if (h->tokf_stage_bytes) cudaFree(h->tokf_stage_bytes);
  if (h->tokf_vec) cudaFree(h->tokf_vec);
  if (h->mel_tables) cudaFree(h->mel_tables);
  if (h->prog_arena) cudaFree(h->prog_arena);
  for (auto& kv : h->ring_tabs) if (kv.second.dev) cudaFree(kv.second.dev);
  if (h->lm_clips) cudaFree(h->lm_clips);
  if (h->ev_lm_clips) cudaEventDestroy(h->ev_lm_clips);
  for (cudaEvent_t e : h->prof.ev) cudaEventDestroy(e);
  if (h->side_stream) cudaStreamDestroy(h->side_stream);
  if (h->side2_stream) cudaStreamDestroy(h->side2_stream);
  if (h->ev_join2) cudaEventDestroy(h->ev_join2);
  for (int i = 0; i < 2; ++i) {
    if (h->tok_stream[i]) cudaStreamDestroy(h->tok_stream[i]);
    if (h->ev_tok_join[i]) cudaEventDestroy(h->ev_tok_join[i]);
  }
  if (h->ev_tok_fork) cudaEventDestroy(h->ev_tok_fork);
  if (h->tail_stream) cudaStreamDestroy(h->tail_stream);
  for (int i = 0; i < 2; ++i) { if (h->ev_front[i]) cudaEventDestroy(h->ev_front[i]); if (h->ev_tail_done[i]) cudaEventDestroy(h->ev_tail_done[i]); }
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_start) cudaEventDestroy(h->ev_start);
  if (h->ev_audio) cudaEventDestroy(h->ev_audio);
  delete h;
}

extern "C" int64_t lsd_launch_count(lsd_handle* h) { return h ? kernel_launches() - h->launches0 : 0; }

// ================================================================================================
// Weights: consume the reference state_dict (SURVEY.md App. B), fold eval BatchNorm (+conv bias).
// ================================================================================================
namespace {

struct HostT {
  const float* data = nullptr;
  int ndim = 0;
  int64_t shape[8] = {0};
  int64_t numel() const { int64_t n = 1; for (int i = 0; i < ndim; ++i) n *= shape[i]; return n; }
};

struct Loader {
  lsd_handle* h;
  std::map<std::string, HostT> t;
  std::vector<float> arena;          // fp32 host staging of the packed device arena
  std::string missing;
  const HostT* get(const std::string& name, std::initializer_list<int64_t> shape) {
    auto it = t.find(name);
    if (it == t.end()) { if (missing.empty()) missing = "missing key " + name; return nullptr; }
    const HostT& x = it->second;
    bool ok = x.ndim == (int)shape.size();
    int i = 0;
    for (int64_t s : shape) { if (ok && x.shape[i] != s) ok = false; ++i; }
    if (!ok) { if (missing.empty()) missing = "shape mismatch for " + name; return nullptr; }
    return &x;
  }
  size_t reserve(size_t n) {  // 64-float (256 B) aligned
    size_t off = (arena.size() + 63) & ~size_t(63);
    arena.resize(off + n, 0.f);
    return off;
  }
};

// Folded conv / linear: weights [tap][Cin][Cout], per-channel scale/shift.
//   bn != "" : scale = gamma/sqrt(var+eps), shift = beta - mean*scale + bias*scale   (App. A)
//   bn == "" : scale = 1 (null), shift = bias
bool pack_conv(Loader& L, const std::string& key, const std::string& wname, const std::string& bname, const std::string& bn,
               int Cout, int Cin, int kt, int kh, int kw) {
  const HostT* w = nullptr;
  if (kt > 0) w = L.get(wname, {Cout, Cin, kt, kh, kw});
  else if (kh > 0) { w = L.get(wname, {Cout, Cin, kh, kw}); kt = 1; }
  else if (kw > 0) { w = L.get(wname, {Cout, Cin, kw}); kt = kh = 1; }
  else { w = L.get(wname, {Cout, Cin}); kt = kh = kw = 1; }
  if (!w) return false;
  const int taps = kt * kh * kw;
  ConvP c;
  c.Cin = Cin; c.Cout = Cout; c.kt = kt; c.kh = kh; c.kw = kw;
  c.w_off = L.reserve((size_t)taps * Cin * Cout);
  for (int co = 0; co < Cout; ++co)
    for (int ci = 0; ci < Cin; ++ci)
      for (int tp = 0; tp < taps; ++tp)
        L.arena[c.w_off + ((size_t)tp * Cin + ci) * Cout + co] = w->data[((size_t)co * Cin + ci) * taps + tp];
  const HostT* b = bname.empty() ? nullptr : L.get(bname, {Cout});
  if (!bname.empty() && !b) return false;
  c.shift_off = L.reserve(Cout);
  c.has_scale = !bn.empty();
  if (c.has_scale) {
    const HostT *g = L.get(bn + ".weight", {Cout}), *be = L.get(bn + ".bias", {Cout}),
                *mu = L.get(bn + ".running_mean", {Cout}), *var = L.get(bn + ".running_var", {Cout});
    if (!g || !be || !mu || !var) return false;
    if (L.t.find(bn + ".num_batches_tracked") == L.t.end()) { L.missing = "missing key " + bn + ".num_batches_tracked"; return false; }
    c.scale_off = L.reserve(Cout);
    for (int i = 0; i < Cout; ++i) {
      const float sc = g->data[i] / sqrtf(var->data[i] + 1e-5f);
      L.arena[c.scale_off + i] = sc;
      L.arena[c.shift_off + i] = be->data[i] - mu->data[i] * sc + (b ? b->data[i] * sc : 0.f);
    }
  } else {
    for (int i = 0; i < Cout; ++i) L.arena[c.shift_off + i] = b ? b->data[i] : 0.f;
  }
  L.h->convs[key] = c;
  return true;
}

bool pack_vec(Loader& L, const std::string& key, const std::string& name, std::initializer_list<int64_t> shape) {
  const HostT* v = L.get(name, shape);
  if (!v) return false;
  const size_t off = L.reserve((size_t)v->numel());
  memcpy(&L.arena[off], v->data, sizeof(float) * v->numel());
  L.h->vecs[key] = off;
  return true;
}

// Cross-attention input projections regrouped by *source* tensor so each source needs one GEMM:
//   from visual tokens: [Q of v2a | K of a2v | V of a2v];  from audio tokens: [Q of a2v | K of v2a | V of v2a]
bool pack_cross_inproj(Loader& L) {
  const HostT *w1 = L.get("cross_modal.v2a_attn.in_proj_weight", {768, 256}), *b1 = L.get("cross_modal.v2a_attn.in_proj_bias", {768}),
              *w2 = L.get("cross_modal.a2v_attn.in_proj_weight", {768, 256}), *b2 = L.get("cross_modal.a2v_attn.in_proj_bias", {768});
  if (!w1 || !b1 || !w2 || !b2) return false;
  for (int side = 0; side < 2; ++side) {
    ConvP c;
    c.Cin = 256; c.Cout = 768; c.kt = c.kh = c.kw = 1; c.has_scale = false;
    c.w_off = L.reserve(256 * 768);
    c.shift_off = L.reserve(768);
    for (int blk = 0; blk < 3; ++blk) {
      // side 0 (visual source): Q from v2a, K/V from a2v;  side 1 (audio source): Q from a2v, K/V from v2a
      const bool from_v2a = (side == 0) ? (blk == 0) : (blk != 0);
      const HostT* w = from_v2a ? w1 : w2;
      const HostT* b = from_v2a ? b1 : b2;
      for (int o = 0; o < 256; ++o) {
        const int src_row = blk * 256 + o;
        L.arena[c.shift_off + blk * 256 + o] = b->data[src_row];
        for (int i = 0; i < 256; ++i) L.arena[c.w_off + (size_t)i * 768 + blk * 256 + o] = w->data[(size_t)src_row * 256 + i];
      }
    }
    L.h->convs[side == 0 ? "cross.in_v" : "cross.in_a"] = c;
  }
  return true;
}

// Projection followed by the cross-attention in-projection is two Linear layers with nothing in between
// (fusion_module.py:108-124 -> :54-66), so the in-projection of a token can be taken straight from the encoder feature:
//   [emb | in_proj(emb)] = feat @ [Wp | Wp Win] + [bp | bp Win + bin]          (one GEMM with 1024 output columns)
// (the audio side applies it to the interpolated features: interpolation along the token axis commutes with a per-token affine
// map).  Products are accumulated in double; "cross.vcomb" / "cross.acomb" are used by the fused token path only.
bool pack_comb_proj(Loader& L, const char* key, const char* proj_key, const char* in_key) {
  const ConvP pr = L.h->convs.at(proj_key), in = L.h->convs.at(in_key);
  ConvP c;
  c.Cin = 256; c.Cout = 1024; c.kt = c.kh = c.kw = 1; c.has_scale = false;
  c.w_off = L.reserve((size_t)256 * 1024);
  c.shift_off = L.reserve(1024);
  std::vector<double> acc(768);
  for (int i = 0; i < 256; ++i) {
    for (int o = 0; o < 256; ++o) L.arena[c.w_off + (size_t)i * 1024 + o] = L.arena[pr.w_off + (size_t)i * 256 + o];
    std::fill(acc.begin(), acc.end(), 0.0);
    for (int k = 0; k < 256; ++k) {
      const double a = L.arena[pr.w_off + (size_t)i * 256 + k];
      const float* row = &L.arena[in.w_off + (size_t)k * 768];
      for (int o = 0; o < 768; ++o) acc[o] += a * (double)row[o];
    }
    for (int o = 0; o < 768; ++o) L.arena[c.w_off + (size_t)i * 1024 + 256 + o] = (float)acc[o];
  }
  for (int o = 0; o < 256; ++o) L.arena[c.shift_off + o] = L.arena[pr.shift_off + o];
  for (int o = 0; o < 768; ++o) {
    double a = L.arena[in.shift_off + o];
    for (int k = 0; k < 256; ++k) a += (double)L.arena[pr.shift_off + k] * (double)L.arena[in.w_off + (size_t)k * 768 + o];
    L.arena[c.shift_off + 256 + o] = (float)a;
  }
  L.h->convs[key] = c;
  return true;
}

}  // namespace

extern "C" int lsd_load_weights(lsd_handle* h, const lsd_tensor* tensors, int n) {
  if (!h || !tensors) return lsd_fail(h, LSD_ERR_ARG, "lsd_load_weights: null argument");
  ENTER_DEVICE(h);
  Loader L;
  L.h = h;
  h->convs.clear();
  h->vecs.clear();
  h->loaded = false;
  for (int i = 0; i < n; ++i) {
    const lsd_tensor& s = tensors[i];
    if (!s.name) return lsd_fail(h, LSD_ERR_ARG, "lsd_load_weights: tensor %d has no name", i);
    if (s.dtype == LSD_I64) { HostT x; x.ndim = 0; L.t[s.name] = x; continue; }  // num_batches_tracked: presence only
    if (s.dtype != LSD_F32 || !s.data) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_load_weights: %s must be fp32 host data", s.name);
    HostT x;
    x.data = reinterpret_cast<const float*>(s.data);
    x.ndim = s.ndim;
    for (int d = 0; d < s.ndim && d < 8; ++d) x.shape[d] = s.shape[d];
    L.t[s.name] = x;
  }
  if (n != 270) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_load_weights: expected the 270-entry reference state_dict, got %d entries", n);
  bool ok = true;
  auto conv3 = [&](const std::string& p, int co, int ci, int kt, int kh, int kw, const std::string& bias = "") {
    ok = ok && pack_conv(L, p, p + ".0.weight", bias, p + ".1", co, ci, kt, kh, kw);
  };
  // visual encoder (visual_encoder.py:113-152)
  conv3("visual_encoder.stem", 64, 3, 3, 7, 7);
  const int chans[4][2] = {{64, 64}, {64, 128}, {128, 256}, {256, 256}};
  for (int l = 0; l < 4; ++l) {
    const std::string p = "visual_encoder.layer" + std::to_string(l + 1);
    conv3(p + ".conv1", chans[l][1], chans[l][0], 3, 3, 3);
    conv3(p + ".conv2", chans[l][1], chans[l][1], 3, 3, 3);
    if (l > 0) conv3(p + ".downsample", chans[l][1], chans[l][0], 1, 1, 1);
  }
  // audio encoder (audio_encoder.py:128-156)
  conv3("audio_encoder.stem", 64, 1, 0, 7, 7);
  for (int l = 0; l < 4; ++l) {
    const std::string p = "audio_encoder.layer" + std::to_string(l + 1);
    conv3(p + ".conv1", chans[l][1], chans[l][0], 0, 3, 3);
    conv3(p + ".conv2", chans[l][1], chans[l][1], 0, 3, 3);
    if (l > 0) conv3(p + ".downsample", chans[l][1], chans[l][0], 0, 1, 1);
  }
  auto linear = [&](const std::string& key, const std::string& p, int co, int ci) {
    ok = ok && pack_conv(L, key, p + ".weight", p + ".bias", "", co, ci, 0, 0, 0);
  };
  linear("projection.visual_proj", "projection.visual_proj", 256, 256);
  linear("projection.audio_proj", "projection.audio_proj", 256, 256);
  ok = ok && pack_cross_inproj(L);
  ok = ok && pack_comb_proj(L, "cross.vcomb", "projection.visual_proj", "cross.in_v") && pack_comb_proj(L, "cross.acomb", "projection.audio_proj", "cross.in_a");
  linear("cross.v2a.out", "cross_modal.v2a_attn.out_proj", 256, 256);
  linear("cross.a2v.out", "cross_modal.a2v_attn.out_proj", 256, 256);
  linear("cross.gate0", "cross_modal.gate.0", 256, 512);
  ok = ok && pack_vec(L, "cross.gate2.w", "cross_modal.gate.2.weight", {1, 256});
  ok = ok && pack_vec(L, "cross.gate2.b", "cross_modal.gate.2.bias", {1});
  linear("cross.fuse", "cross_modal.fuse.0", 256, 256);
  // temporal transformer (temporal.py:31-77)
  ok = ok && pack_vec(L, "temporal.cls", "temporal.cls_token", {1, 1, 256});
  for (int k : {3, 5, 7}) {
    const std::string p = "temporal.branch_k" + std::to_string(k);
    ok = ok && pack_conv(L, p, p + ".0.weight", "", p + ".1", 256, 256, 0, 0, k);
  }
  linear("temporal.pre_scale_proj", "temporal.pre_scale_proj", 256, 768);
  for (int l = 0; l < 4; ++l) {
    const std::string p = "temporal.transformer.layers." + std::to_string(l);
    const std::string k = "t" + std::to_string(l);
    ok = ok && pack_conv(L, k + ".in", p + ".self_attn.in_proj_weight", p + ".self_attn.in_proj_bias", "", 768, 256, 0, 0, 0);
    linear(k + ".out", p + ".self_attn.out_proj", 256, 256);
    linear(k + ".ff1", p + ".linear1", 1024, 256);
    linear(k + ".ff2", p + ".linear2", 256, 1024);
    ok = ok && pack_vec(L, k + ".ln1.w", p + ".norm1.weight", {256}) && pack_vec(L, k + ".ln1.b", p + ".norm1.bias", {256});
    ok = ok && pack_vec(L, k + ".ln2.w", p + ".norm2.weight", {256}) && pack_vec(L, k + ".ln2.b", p + ".norm2.bias", {256});
  }
  // artifact detector (artifact_detector.py:33-43,74-93,142-147)
  const std::string td = "artifact_detector.temporal_detector.temporal_conv";
  ok = ok && pack_conv(L, "art.td0", td + ".0.weight", td + ".0.bias", td + ".1", 128, 256, 3, 3, 3);
  ok = ok && pack_conv(L, "art.td3", td + ".3.weight", td + ".3.bias", td + ".4", 64, 128, 3, 3, 3);
  const std::string hf = "artifact_detector.high_freq_detector";
  ok = ok && pack_conv(L, "art.lap", hf + ".laplacian.weight", "", "", 3, 3, 0, 3, 3);
  ok = ok && pack_conv(L, "art.hf0", hf + ".conv3d.0.weight", hf + ".conv3d.0.bias", hf + ".conv3d.1", 32, 3, 3, 3, 3);
  ok = ok && pack_conv(L, "art.hf3", hf + ".conv3d.3.weight", hf + ".conv3d.3.bias", hf + ".conv3d.4", 64, 32, 3, 3, 3);
  linear("art.fuse0", "artifact_detector.artifact_fusion.0", 256, 448);
  linear("art.fuse2", "artifact_detector.artifact_fusion.2", 128, 256);
  // head (classifier.py:14-20)
  linear("head.fc0", "classifier.net.0", 128, 384);
  ok = ok && pack_vec(L, "head.ln.w", "classifier.net.3.weight", {128}) && pack_vec(L, "head.ln.b", "classifier.net.3.bias", {128});
  ok = ok && pack_vec(L, "head.out.w", "classifier.net.4.weight", {1, 128}) && pack_vec(L, "head.out.b", "classifier.net.4.bias", {1});
  if (!ok) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_load_weights: %s", L.missing.empty() ? "pack failed" : L.missing.c_str());

  if (h->warena) { cudaFree(h->warena); h->warena = nullptr; }
  CUDA_OK(h, cudaMalloc(&h->warena, L.arena.size() * sizeof(float)));
  CUDA_OK(h, cudaMemcpy(h->warena, L.arena.data(), L.arena.size() * sizeof(float), cudaMemcpyHostToDevice));
  int rc = pack_bf16_weights(h, L.arena);
  if (rc != 0) return rc;
  h->loaded = true;
  ++h->generation;
  return LSD_OK;
}

// ================================================================================================
// Workspace plan
// ================================================================================================
using namespace lsdfw;

namespace {
int check_dtype(lsd_handle* h, int dt, const char* what) {
  if (dt < LSD_F32 || dt > LSD_U8) return lsd_fail(h, LSD_ERR_ARG, "%s: unsupported dtype %d", what, dt);
  return 0;
}

// First mel column of an audio window of Ta columns that must end inside the clip (predictor.py:540-547): past the end -> the
// last full window, then never before column 0.
long clamp_audio_start(long a_start, int Ta, int Ta_full) {
  if (a_start + Ta > Ta_full) a_start = Ta_full - Ta;
  return a_start < 0 ? 0 : a_start;
}

// Base audio start of window i: explicit, or a_start = int(round(v_start * a_ratio)) (round-half-even), clamped
long base_audio_start(const int32_t* starts_host, const int32_t* audio_starts_host, int i, int Ta, int Ta_full, int total_v_frames) {
  const double a_ratio = (double)Ta_full / (double)(total_v_frames > 1 ? total_v_frames : 1);
  const long a = audio_starts_host ? (long)audio_starts_host[i] : (long)nearbyint((double)starts_host[i] * a_ratio);
  return clamp_audio_start(a, Ta, Ta_full);
}

// dst row r = src row r, `width` 2-byte units per row (the per-variant route of the audio-variant entry points)
__global__ void copy_rows_u16_kernel(const uint16_t* __restrict__ src, int64_t src_ld, uint16_t* __restrict__ dst, int64_t dst_ld,
                                     int rows, int64_t width) {
  const int64_t n = (int64_t)rows * width;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / width, c = i - r * width;
    dst[r * dst_ld + c] = src[r * src_ld + c];
  }
}
void copy_rows_bytes(const void* src, int64_t src_ld, void* dst, int64_t dst_ld, int rows, int64_t width, cudaStream_t st) {
  const int64_t n = (int64_t)rows * (width / 2);
  const int grid = (int)std::min<int64_t>((n + 255) / 256, 4096);
  copy_rows_u16_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const uint16_t*>(src), src_ld / 2, reinterpret_cast<uint16_t*>(dst), dst_ld / 2,
                                             rows, width / 2);
  count_launch();
}
size_t align256(size_t n) { return (n + 255) & ~size_t(255); }

}  // namespace

extern "C" int lsd_audio_tokens(int Ta) {
  if (Ta < 1) return 0;
  return osz(osz(osz(Ta, 7, 2, 3), 3, 2, 1), 3, 2, 1);
}

extern "C" size_t lsd_workspace_bytes(lsd_handle* h, int B, int T, int H, int W, int F, int Ta, int precision) {
  Shapes s;
  if (make_shapes(h, B, T, H, W, F, Ta, s) != 0) return 0;
  Plan p;
  if (precision == LSD_PREC_BF16) make_plan_bf16(h, s.B, s.T, s.H, s.W, s.F, s.Ta, p.stages, p.cursor);
  else make_plan_f32(s, p);
  return p.cursor + 256;
}

extern "C" int lsd_forward(lsd_handle* h, const void* video, int video_dtype, int video_layout, const void* audio, int audio_dtype,
                           int B, int T, int H, int W, int F, int Ta, int precision, float* logits_out, const lsd_aux* aux,
                           void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_forward: no weights loaded (call lsd_load_weights first)");
  Shapes s;
  int rc = make_shapes(h, B, T, H, W, F, Ta, s);
  if (rc) return rc;
  if (B == 0) return LSD_OK;
  if (!video || !audio || !logits_out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_forward: null pointer argument");
  if ((rc = check_dtype(h, video_dtype, "video")) || (rc = check_dtype(h, audio_dtype, "audio"))) return rc;
  if (audio_dtype == LSD_U8) return lsd_fail(h, LSD_ERR_ARG, "audio: uint8 log-mel is not supported");
  if (video_layout != LSD_NCDHW && video_layout != LSD_NDHWC) return lsd_fail(h, LSD_ERR_ARG, "bad video layout %d", video_layout);
  if (precision != LSD_PREC_FP32 && precision != LSD_PREC_BF16) return lsd_fail(h, LSD_ERR_ARG, "bad precision %d", precision);
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (precision == LSD_PREC_BF16) {
    rc = forward_bf16(h, B, T, H, W, F, Ta, video, video_dtype, video_layout, audio, audio_dtype, logits_out, aux,
                      reinterpret_cast<char*>(workspace), workspace_bytes, st, false);
    if (rc) return rc;
  } else {
    Plan p;
    make_plan_f32(s, p);
    if (p.cursor > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", p.cursor, workspace_bytes);
    h->stages = p.stages;
    for (WsSig& w : h->ws_sig) w.ptr = nullptr;  // the fp32 plan overwrites any bf16 zero padding kept in this workspace
    rc = forward_f32(h, s, p, reinterpret_cast<char*>(workspace), aux, logits_out, st, false, video, video_dtype, video_layout, audio, audio_dtype);
    if (rc) return rc;
  }
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

// ================================================================================================
// Window builder + batched scoring (replaces the serial loop of Predictor._run_chunked_inference)
// ================================================================================================
extern "C" size_t lsd_score_workspace_bytes(lsd_handle* h, int batch, int T, int H, int W, int F, int Ta, int precision) {
  const size_t fw = lsd_workspace_bytes(h, batch, T, H, W, F, Ta, precision);
  if (fw == 0) return 0;
  return fw + 2 * (((size_t)batch * sizeof(int32_t) + 255) & ~size_t(255)) + 256;
}

namespace {
// Returns the track a batch of rows [r0, r0+nb) reads, after enqueueing on `st` whatever builds it (score_window_variants: the
// batch's pseudo-track).  Empty: every batch reads the caller's track.
using BatchTrack = std::function<int(int r0, int nb, const uint8_t*& track, int& n_frames)>;

// The batch loop of lsd_score_windows, shared with score_window_variants.  h->idx_host holds the first track frame of row r at [r]
// and its first mel column at [n_rows + r]; the caller has checked every argument and the workspace size.  feats_out (optional):
// row r receives the head's input row of row r, [cls | comb[:, 256:448]] (LSD_BRANCH_FEATURES floats).
int score_rows(lsd_handle* h, const uint8_t* track, int n_frames, int n_rows, int T, int H, int W, const float* mel_full, int F,
               int Ta_full, int Ta, int precision, int batch, float* logits_out, void* workspace, size_t workspace_bytes,
               cudaStream_t st, const BatchTrack& batch_track, float* feats_out = nullptr) {
  int rc = 0;
  const size_t idx_bytes = ((size_t)batch * sizeof(int32_t) + 255) & ~size_t(255);
  char* ws = reinterpret_cast<char*>(workspace);
  int32_t* d_vs = reinterpret_cast<int32_t*>(ws);
  int32_t* d_as = reinterpret_cast<int32_t*>(ws + idx_bytes);
  char* fws = ws + 2 * idx_bytes;
  // Cross-batch pipelining (tensor-core route, more than one batch, workspace >= 2 x lsd_score_workspace_bytes): batches
  // alternate between the two halves of the workspace; the tail of batch k (audio encoder, token path, head, artifact branch)
  // runs on side streams while this stream continues with the visual encoder of batch k+1.
  const size_t fw_bytes = ((lsd_workspace_bytes(h, batch, T, H, W, F, Ta, precision) + 255) & ~size_t(255));
  const bool pipelined = precision == LSD_PREC_BF16 && n_rows > batch && workspace_bytes >= 2 * idx_bytes + 2 * fw_bytes &&
                         getenv("LSD_NO_PIPELINE") == nullptr;
  if (pipelined && (rc = ensure_pipeline(h))) return rc;
  int k = 0;
  for (int w0 = 0; w0 < n_rows; w0 += batch, ++k) {
    const int nb = (n_rows - w0) < batch ? (n_rows - w0) : batch;
    const int parity = k & 1;
    if (pipelined && k >= 2) CUDA_OK(h, cudaStreamWaitEvent(st, h->ev_tail_done[parity], 0));   // this half of the workspace is free again
    CUDA_OK(h, cudaMemcpyAsync(d_vs, &h->idx_host[w0], nb * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CUDA_OK(h, cudaMemcpyAsync(d_as, &h->idx_host[n_rows + w0], nb * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (batch_track && (rc = batch_track(w0, nb, track, n_frames))) return rc;
    float* feats_b = feats_out ? feats_out + (size_t)w0 * LSD_BRANCH_FEATURES : nullptr;
    if (precision == LSD_PREC_BF16) {
      if (pipelined) rc = score_batch_bf16(h, track, n_frames, d_vs, d_as, mel_full, Ta_full, nb, T, H, W, F, Ta, logits_out + w0,
                                           fws + (size_t)parity * fw_bytes, fw_bytes, st, parity, feats_b);
      else rc = score_batch_bf16(h, track, n_frames, d_vs, d_as, mel_full, Ta_full, nb, T, H, W, F, Ta, logits_out + w0, fws,
                                 workspace_bytes - 2 * idx_bytes, st, -1, feats_b);
      if (rc) return rc;
    } else {
      Shapes sb;
      make_shapes(h, nb, T, H, W, F, Ta, sb);
      Plan pb;
      make_plan_f32(sb, pb);
      h->stages = pb.stages;
      for (WsSig& w : h->ws_sig) w.ptr = nullptr;
      Ctx c{h, fws, &pb, st};
      launch_gather_windows_u8(track, n_frames, d_vs, c.buf("vid"), nb, T, H * W * 3, st);
      launch_gather_audio(mel_full, F, Ta_full, d_as, c.buf("aud"), nb, Ta, st);
      rc = forward_f32(h, sb, pb, fws, nullptr, logits_out + w0, st, true, nullptr, 0, 0, nullptr, 0);
      if (rc) return rc;
      // comb holds the whole head input row here: [cls (a copy of the token rows) | raw | delta | hf]
      if (feats_b) CUDA_OK(h, cudaMemcpyAsync(feats_b, c.buf("comb"), (size_t)nb * LSD_BRANCH_FEATURES * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
  }
  if (pipelined) {   // the caller's stream sees every batch's logits
    CUDA_OK(h, cudaStreamWaitEvent(st, h->ev_tail_done[0], 0));
    if (k >= 2) CUDA_OK(h, cudaStreamWaitEvent(st, h->ev_tail_done[1], 0));
  }
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

int check_windows(lsd_handle* h, const int32_t* starts_host, int n_windows, int T, int n_frames) {
  for (int i = 0; i < n_windows; ++i)
    if (starts_host[i] < 0 || starts_host[i] + T > n_frames)
      return lsd_fail(h, LSD_ERR_SHAPE, "window %d [%d,%d) is outside the %d-frame track", i, starts_host[i], starts_host[i] + T, n_frames);
  return 0;
}
}  // namespace

namespace {
// lsd_score_windows and lsd_score_branch_features (feats_out != nullptr)
int score_windows(lsd_handle* h, const char* fn, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                  const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full, int total_v_frames, int Ta,
                  int precision, int batch, float* logits_out, float* feats_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "%s: no weights loaded", fn);
  if (n_windows == 0) return LSD_OK;
  if (!track || !starts_host || !mel_full || !logits_out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "%s: null pointer argument", fn);
  if (batch < 1 || n_windows < 0 || n_frames < 1 || Ta_full < 1) return lsd_fail(h, LSD_ERR_SHAPE, "%s: bad extents", fn);
  if (precision != LSD_PREC_FP32 && precision != LSD_PREC_BF16) return lsd_fail(h, LSD_ERR_ARG, "bad precision %d", precision);
  Shapes s;
  int rc = make_shapes(h, batch, T, H, W, F, Ta, s);
  if (rc) return rc;
  if ((rc = check_windows(h, starts_host, n_windows, T, n_frames))) return rc;
  ENTER_DEVICE(h);
  const size_t need = lsd_score_workspace_bytes(h, batch, T, H, W, F, Ta, precision);
  if (need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  // all window/audio starts are staged once (pinned-free small copies are ordered on the stream)
  h->idx_host.resize((size_t)2 * n_windows);
  for (int i = 0; i < n_windows; ++i) {
    h->idx_host[i] = starts_host[i];
    h->idx_host[n_windows + i] = (int32_t)base_audio_start(starts_host, audio_starts_host, i, Ta, Ta_full, total_v_frames);
  }
  return score_rows(h, track, n_frames, n_windows, T, H, W, mel_full, F, Ta_full, Ta, precision, batch, logits_out, workspace,
                    workspace_bytes, reinterpret_cast<cudaStream_t>(stream), BatchTrack(), feats_out);
}
}  // namespace

extern "C" int lsd_score_windows(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                                 const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full, int total_v_frames, int Ta,
                                 int precision, int batch, float* logits_out, void* workspace, size_t workspace_bytes, void* stream) {
  return score_windows(h, "lsd_score_windows", track, n_frames, H, W, starts_host, audio_starts_host, n_windows, T, mel_full, F, Ta_full,
                       total_v_frames, Ta, precision, batch, logits_out, nullptr, workspace, workspace_bytes, stream);
}

// ================================================================================================
// Branch attribution (attribution.cu): the head's input rows out of the plain scoring loop, then exact Shapley values of its
// four inputs against a background set
// ================================================================================================
extern "C" int lsd_score_branch_features(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                                         const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                                         int total_v_frames, int Ta, int precision, int batch, float* logits_out, float* feats_out,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  if (h && h->loaded && n_windows > 0 && !feats_out) return lsd_fail(h, LSD_ERR_ARG, "lsd_score_branch_features: feats_out is NULL");
  return score_windows(h, "lsd_score_branch_features", track, n_frames, H, W, starts_host, audio_starts_host, n_windows, T, mel_full, F,
                       Ta_full, total_v_frames, Ta, precision, batch, logits_out, feats_out, workspace, workspace_bytes, stream);
}

namespace {
// Workspace: [projections of the n window rows and M background rows | per-(window, mask, chunk) logit sums | v(15) per window]
bool attribution_extents_ok(int n, int M) {
  return n >= 0 && M >= 1 && M <= LSD_MAX_BACKGROUND && (int64_t)n * (15 * (int64_t)M + 1) <= INT32_MAX;
}
size_t attribution_partial_floats(int n, int M) { return (size_t)n * 15 * ((M + ATTR_CHUNK - 1) / ATTR_CHUNK); }
}  // namespace

extern "C" size_t lsd_branch_attribution_workspace_bytes(int n, int M) {
  if (!attribution_extents_ok(n, M)) return 0;
  return align256(((size_t)n + M) * ATTR_PROJ * sizeof(float)) + align256(attribution_partial_floats(n, M) * sizeof(float)) +
         align256((size_t)n * sizeof(float)) + 256;
}

extern "C" int lsd_branch_attribution(lsd_handle* h, const float* feats, int n, const float* background, int M, float* values_out,
                                      float* phi_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!feats || !background || !values_out || !phi_out || !workspace)
    return lsd_fail(h, LSD_ERR_ARG, "lsd_branch_attribution: null pointer argument");
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_branch_attribution: no weights loaded");
  if (!attribution_extents_ok(n, M))
    return lsd_fail(h, LSD_ERR_SHAPE, "lsd_branch_attribution: n = %d windows, M = %d background rows: expected n >= 0, 1 <= M <= %d and "
                    "n*(15M+1) <= INT32_MAX", n, M, LSD_MAX_BACKGROUND);
  const size_t need = lsd_branch_attribution_workspace_bytes(n, M);
  if (need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  if (n == 0) return LSD_OK;
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  float* proj = reinterpret_cast<float*>(ws);
  float* partial = reinterpret_cast<float*>(ws + align256(((size_t)n + M) * ATTR_PROJ * sizeof(float)));
  float* v15 = partial + align256(attribution_partial_floats(n, M) * sizeof(float)) / sizeof(float);
  lsd::HeadW hw;
  auto cw = [&](const char* key) { return h->warena + h->convs.at(key).w_off; };
  auto cb = [&](const char* key) { return h->warena + h->convs.at(key).shift_off; };
  hw.w0 = cw("art.fuse0"); hw.b0 = cb("art.fuse0"); hw.w2 = cw("art.fuse2"); hw.b2 = cb("art.fuse2");
  hw.wc = cw("head.fc0"); hw.bc = cb("head.fc0");
  hw.lng = h->warena + h->vecs.at("head.ln.w"); hw.lnb = h->warena + h->vecs.at("head.ln.b");
  hw.wo = h->warena + h->vecs.at("head.out.w"); hw.bo = h->warena + h->vecs.at("head.out.b");
  launch_branch_attribution(feats, n, background, M, hw, proj, partial, v15, values_out, phi_out, h->num_sms, st);
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

// ================================================================================================
// Window variants: K device-built copies of every window (occlusion.cu, warp.cu, jpeg.cu, resize.cu, retime.cu), scored by the batch
// loop of lsd_score_windows
// ================================================================================================
// Workspace: [variant tables | track starts of one batch's windows | pseudo-track of `batch` built windows | lsd_score_windows
// workspace].  The pseudo-track is read only by the batch's first kernel on the caller's stream (the tensor-core pixel rows or the
// fp32 gather), so one copy serves pipelined batches too.
namespace {
size_t variant_extra_bytes(size_t table_bytes, int batch, int T, int H, int W) {
  return align256(table_bytes) + align256(((size_t)batch + 1) * sizeof(int32_t)) + align256((size_t)batch * T * H * W * 3);
}

size_t variant_workspace_bytes(lsd_handle* h, size_t table_bytes, int batch, int T, int H, int W, int F, int Ta, int precision) {
  const size_t sw = lsd_score_workspace_bytes(h, batch, T, H, W, F, Ta, precision);
  if (sw == 0) return 0;
  return variant_extra_bytes(table_bytes, batch, T, H, W) + align256(sw);
}

// Enqueues on `st` the kernel that writes rows r0 .. r0+nb-1 (window r / K, variant r % K) into `pseudo`; d_tabs: the variant
// tables, d_wins: the track starts of windows r0 / K, r0 / K + 1, ...
using VariantBuilder = std::function<void(const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* pseudo, cudaStream_t st)>;

// The common part of lsd_score_occlusions / lsd_score_warps / lsd_score_jpeg / lsd_score_resizes / lsd_score_retimes, after each has checked its variants: the remaining
// argument checks, the row table (row r reads frames (r % batch) * T .. of the batch's pseudo-track and the audio slice of window
// r / K), one copy of the K variants' tables (`table_bytes` of them, from tables_host; their region is table_region bytes) and the
// per-batch hook that copies the batch's window starts and runs `build`.  `what` names the variants in messages.
int score_window_variants(lsd_handle* h, const char* fn, const char* what, const uint8_t* track, int n_frames, int H, int W,
                          const int32_t* starts_host, const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F,
                          int Ta_full, int total_v_frames, int Ta, int K, int precision, int batch, float* logits_out, void* workspace,
                          size_t workspace_bytes, void* stream, const void* tables_host, size_t table_bytes, size_t table_region,
                          const VariantBuilder& build) {
  if (n_windows == 0) return LSD_OK;
  if (!track || !starts_host || !mel_full || !logits_out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "%s: null pointer argument", fn);
  if (batch < 1 || n_windows < 0 || n_frames < 1 || Ta_full < 1) return lsd_fail(h, LSD_ERR_SHAPE, "%s: bad extents", fn);
  if ((int64_t)n_windows * K > INT32_MAX) return lsd_fail(h, LSD_ERR_SHAPE, "%d windows x %d %s: too many rows for one call", n_windows, K, what);
  if (precision != LSD_PREC_FP32 && precision != LSD_PREC_BF16) return lsd_fail(h, LSD_ERR_ARG, "bad precision %d", precision);
  Shapes s;
  int rc = make_shapes(h, batch, T, H, W, F, Ta, s);
  if (rc) return rc;
  if ((rc = check_windows(h, starts_host, n_windows, T, n_frames))) return rc;
  const size_t need = variant_workspace_bytes(h, table_region, batch, T, H, W, F, Ta, precision);
  if (need == 0 || need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int n_rows = n_windows * K;
  h->idx_host.resize((size_t)2 * n_rows);
  for (int i = 0; i < n_windows; ++i) {
    const int32_t a = (int32_t)base_audio_start(starts_host, audio_starts_host, i, Ta, Ta_full, total_v_frames);
    for (int k = 0; k < K; ++k) {
      const int r = i * K + k;
      h->idx_host[r] = (r % batch) * T;
      h->idx_host[n_rows + r] = a;
    }
  }
  char* ws = reinterpret_cast<char*>(workspace);
  int32_t* d_tabs = reinterpret_cast<int32_t*>(ws);
  int32_t* d_wins = reinterpret_cast<int32_t*>(ws + align256(table_region));
  uint8_t* pseudo = reinterpret_cast<uint8_t*>(d_wins) + align256(((size_t)batch + 1) * sizeof(int32_t));
  const size_t extra = variant_extra_bytes(table_region, batch, T, H, W);
  CUDA_OK(h, cudaMemcpyAsync(d_tabs, tables_host, table_bytes, cudaMemcpyHostToDevice, st));
  const BatchTrack built = [&](int r0, int nb, const uint8_t*& trk, int& nf) -> int {
    const int wa = r0 / K, wb = (r0 + nb - 1) / K;
    CUDA_OK(h, cudaMemcpyAsync(d_wins, starts_host + wa, (size_t)(wb - wa + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    build(d_tabs, d_wins, r0, nb, pseudo, st);
    trk = pseudo;
    nf = nb * T;
    return 0;
  };
  return score_rows(h, pseudo, batch * T, n_rows, T, H, W, mel_full, F, Ta_full, Ta, precision, batch, logits_out, ws + extra,
                    workspace_bytes - extra, st, built);
}

// The variant tables and the window starts of the entries that return the built windows themselves (lsd_warp_windows,
// lsd_jpeg_windows, lsd_resize_windows, lsd_retime_windows): one launch over all n_windows x K rows into the caller's buffer.
int build_window_variants(lsd_handle* h, const int32_t* starts_host, int n_windows, int K, void* workspace, void* stream,
                          const void* tables_host, size_t table_bytes, uint8_t* out, const VariantBuilder& build) {
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int32_t* d_tabs = reinterpret_cast<int32_t*>(workspace);
  int32_t* d_wins = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(workspace) + align256(table_bytes));
  CUDA_OK(h, cudaMemcpyAsync(d_tabs, tables_host, table_bytes, cudaMemcpyHostToDevice, st));
  CUDA_OK(h, cudaMemcpyAsync(d_wins, starts_host, (size_t)n_windows * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  build(d_tabs, d_wins, 0, n_windows * K, out, st);
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

size_t built_windows_workspace_bytes(size_t table_bytes, int n_windows) {
  return align256(table_bytes) + align256((size_t)n_windows * sizeof(int32_t));
}

constexpr size_t OCCLUSION_TABLE_BYTES = (size_t)LSD_MAX_OCCLUSIONS * 7 * sizeof(int32_t);
}  // namespace

// ------------------------------------------------------------------------------------------------
// Occlusion evidence: K occluded copies of every window (occlusion.cu)
// ------------------------------------------------------------------------------------------------
extern "C" size_t lsd_score_occlusions_workspace_bytes(lsd_handle* h, int batch, int T, int H, int W, int F, int Ta, int precision) {
  if (batch < 1) return 0;
  return variant_workspace_bytes(h, OCCLUSION_TABLE_BYTES, batch, T, H, W, F, Ta, precision);
}

extern "C" int lsd_score_occlusions(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                                    const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                                    int total_v_frames, int Ta, const lsd_occlusion* boxes, int K, int fill, int precision, int batch,
                                    float* logits_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_score_occlusions: no weights loaded");
  if (!boxes) return lsd_fail(h, LSD_ERR_ARG, "lsd_score_occlusions: boxes is NULL");
  if (K < 1 || K > LSD_MAX_OCCLUSIONS) return lsd_fail(h, LSD_ERR_SHAPE, "K = %d occlusion boxes: expected 1 <= K <= %d", K, LSD_MAX_OCCLUSIONS);
  if (fill < 0 || fill > 255) return lsd_fail(h, LSD_ERR_ARG, "lsd_score_occlusions: fill %d is not a uint8 value", fill);
  for (int k = 0; k < K; ++k) {
    const lsd_occlusion& b = boxes[k];
    if (b.t0 < 0 || b.t0 > b.t1 || b.t1 > T || b.y0 < 0 || b.y0 > b.y1 || b.y1 > H || b.x0 < 0 || b.x0 > b.x1 || b.x1 > W)
      return lsd_fail(h, LSD_ERR_SHAPE, "box %d [%d,%d)x[%d,%d)x[%d,%d) is not inside the %dx%dx%d window", k, b.t0, b.t1, b.y0, b.y1,
                      b.x0, b.x1, T, H, W);
    if (b.src < -1 || b.src >= T) return lsd_fail(h, LSD_ERR_SHAPE, "box %d: src %d is outside -1..%d", k, b.src, T - 1);
  }
  static_assert(sizeof(lsd_occlusion) == 7 * sizeof(int32_t), "lsd_occlusion is seven packed int32");
  const VariantBuilder occlude = [&](const int32_t* d_boxes, const int32_t* d_wins, int r0, int nb, uint8_t* pseudo, cudaStream_t st) {
    launch_occlude_windows(track, d_wins, d_boxes, K, r0, nb, T, H, W, fill, pseudo, st);
  };
  return score_window_variants(h, "lsd_score_occlusions", "boxes", track, n_frames, H, W, starts_host, audio_starts_host, n_windows, T,
                               mel_full, F, Ta_full, total_v_frames, Ta, K, precision, batch, logits_out, workspace, workspace_bytes,
                               stream, boxes, (size_t)K * sizeof(lsd_occlusion), OCCLUSION_TABLE_BYTES, occlude);
}

// ------------------------------------------------------------------------------------------------
// Crop-jitter robustness: K re-cropped copies of every window (warp.cu); tables K*T*2(H+W) int32
// ------------------------------------------------------------------------------------------------
namespace {
// The checks every warp entry makes before any GPU work; on success h->variant_tab_host holds the tables of the K*T matrices.
int warp_tables_checked(lsd_handle* h, const char* fn, const lsd_warp* warps, int K, int T, int H, int W) {
  if (!warps) return lsd_fail(h, LSD_ERR_ARG, "%s: warps is NULL", fn);
  if (K < 1 || K > LSD_MAX_WARPS) return lsd_fail(h, LSD_ERR_SHAPE, "K = %d warp variants: expected 1 <= K <= %d", K, LSD_MAX_WARPS);
  if (T < 1 || H < 1 || W < 1 || (int64_t)H * W * 3 > INT32_MAX || !warp_extents_ok(H, W))
    return lsd_fail(h, LSD_ERR_SHAPE, "%s: bad window extents T=%d H=%d W=%d", fn, T, H, W);
  static_assert(sizeof(lsd_warp) == 6 * sizeof(double), "lsd_warp is six packed doubles");
  h->variant_tab_host.resize(warp_tables_ints(K, T, H, W));
  int bad = 0;
  const int rc = warp_tables(reinterpret_cast<const double*>(warps), K * T, H, W, h->variant_tab_host.data(), &bad);
  if (rc == -1)
    return lsd_fail(h, LSD_ERR_ARG, "warp %d (variant %d, frame %d) has a non-finite entry or is singular", bad, bad / T, bad % T);
  if (rc == -2)
    return lsd_fail(h, LSD_ERR_SHAPE, "warp %d (variant %d, frame %d) maps the %dx%d frame beyond +-32767 px", bad, bad / T, bad % T, H, W);
  return 0;
}
}  // namespace

extern "C" size_t lsd_score_warps_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision) {
  if (batch < 1 || K < 1 || K > LSD_MAX_WARPS) return 0;
  return variant_workspace_bytes(h, warp_tables_ints(K, T, H, W) * sizeof(int32_t), batch, T, H, W, F, Ta, precision);
}

extern "C" int lsd_score_warps(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                               const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                               int total_v_frames, int Ta, const lsd_warp* warps, int K, int precision, int batch, float* logits_out,
                               void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_score_warps: no weights loaded");
  const int rc = warp_tables_checked(h, "lsd_score_warps", warps, K, T, H, W);
  if (rc) return rc;
  const size_t tab_bytes = h->variant_tab_host.size() * sizeof(int32_t);
  const VariantBuilder warp = [&](const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* pseudo, cudaStream_t st) {
    launch_warp_windows(track, d_wins, d_tabs, K, r0, nb, T, H, W, pseudo, st);
  };
  return score_window_variants(h, "lsd_score_warps", "warps", track, n_frames, H, W, starts_host, audio_starts_host, n_windows, T,
                               mel_full, F, Ta_full, total_v_frames, Ta, K, precision, batch, logits_out, workspace, workspace_bytes,
                               stream, h->variant_tab_host.data(), tab_bytes, tab_bytes, warp);
}

// The warped windows themselves, written to a caller buffer by the builder lsd_score_warps uses: what the K variants look like.
extern "C" size_t lsd_warp_windows_workspace_bytes(int n_windows, int K, int T, int H, int W) {
  if (n_windows < 1 || K < 1 || K > LSD_MAX_WARPS || T < 1 || H < 1 || W < 1) return 0;
  return built_windows_workspace_bytes(warp_tables_ints(K, T, H, W) * sizeof(int32_t), n_windows);
}

extern "C" int lsd_warp_windows(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host, int n_windows,
                                int T, const lsd_warp* warps, int K, uint8_t* out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  int rc = warp_tables_checked(h, "lsd_warp_windows", warps, K, T, H, W);
  if (rc) return rc;
  if (n_windows == 0) return LSD_OK;
  if (!track || !starts_host || !out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_warp_windows: null pointer argument");
  if (n_windows < 0 || n_frames < 1) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_warp_windows: bad extents");
  if ((int64_t)n_windows * K * T > INT32_MAX) return lsd_fail(h, LSD_ERR_SHAPE, "%d windows x %d warps: too many frames for one call", n_windows, K);
  if ((rc = check_windows(h, starts_host, n_windows, T, n_frames))) return rc;
  const size_t need = lsd_warp_windows_workspace_bytes(n_windows, K, T, H, W);
  if (need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  const VariantBuilder warp = [&](const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* o, cudaStream_t st) {
    launch_warp_windows(track, d_wins, d_tabs, K, r0, nb, T, H, W, o, st);
  };
  return build_window_variants(h, starts_host, n_windows, K, workspace, stream, h->variant_tab_host.data(),
                               h->variant_tab_host.size() * sizeof(int32_t), out, warp);
}

// ------------------------------------------------------------------------------------------------
// Compression robustness: K JPEG round-tripped copies of every window (jpeg.cu); tables JPEG_TAB_INTS int32 per variant
// ------------------------------------------------------------------------------------------------
namespace {
// The checks every JPEG entry makes before any GPU work; on success h->variant_tab_host holds the K variants' tables and *any444
// tells whether one samples 4:4:4.
int jpeg_tables_checked(lsd_handle* h, const char* fn, const lsd_jpeg* v, int K, int channel_order, int T, int H, int W, bool* any444) {
  if (!v) return lsd_fail(h, LSD_ERR_ARG, "%s: variants is NULL", fn);
  if (K < 1 || K > LSD_MAX_JPEG_VARIANTS)
    return lsd_fail(h, LSD_ERR_SHAPE, "K = %d JPEG variants: expected 1 <= K <= %d", K, LSD_MAX_JPEG_VARIANTS);
  if (channel_order != LSD_RGB && channel_order != LSD_BGR) return lsd_fail(h, LSD_ERR_ARG, "%s: bad channel order %d", fn, channel_order);
  bool any420 = false;
  *any444 = false;
  for (int k = 0; k < K; ++k) {
    if (v[k].sampling != LSD_JPEG_NONE && v[k].sampling != LSD_JPEG_444 && v[k].sampling != LSD_JPEG_420)
      return lsd_fail(h, LSD_ERR_ARG, "JPEG variant %d: bad sampling %d", k, v[k].sampling);
    if (v[k].sampling != LSD_JPEG_NONE && (v[k].quality < 1 || v[k].quality > 100))
      return lsd_fail(h, LSD_ERR_ARG, "JPEG variant %d: quality %d is outside 1..100", k, v[k].quality);
    any420 |= v[k].sampling == LSD_JPEG_420;
    *any444 |= v[k].sampling == LSD_JPEG_444;
  }
  const int mcu = any420 ? 16 : 8;
  if (T < 1 || H < 1 || W < 1 || H % mcu || W % mcu || !jpeg_extents_ok(H, W, *any444))
    return lsd_fail(h, LSD_ERR_SHAPE, "%s: bad window extents T=%d H=%d W=%d (sides multiples of %d, planes within shared memory)", fn, T,
                    H, W, mcu);
  static_assert(sizeof(lsd_jpeg) == 2 * sizeof(int32_t), "lsd_jpeg is two packed int32");
  h->variant_tab_host.resize((size_t)K * JPEG_TAB_INTS);
  jpeg_tables(reinterpret_cast<const int32_t*>(v), K, h->variant_tab_host.data());
  return 0;
}
}  // namespace

extern "C" size_t lsd_score_jpeg_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision) {
  if (batch < 1 || K < 1 || K > LSD_MAX_JPEG_VARIANTS) return 0;
  return variant_workspace_bytes(h, (size_t)K * JPEG_TAB_INTS * sizeof(int32_t), batch, T, H, W, F, Ta, precision);
}

extern "C" int lsd_score_jpeg(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                              const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                              int total_v_frames, int Ta, const lsd_jpeg* variants, int K, int channel_order, int precision, int batch,
                              float* logits_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_score_jpeg: no weights loaded");
  bool any444 = false;
  const int rc = jpeg_tables_checked(h, "lsd_score_jpeg", variants, K, channel_order, T, H, W, &any444);
  if (rc) return rc;
  const size_t tab_bytes = h->variant_tab_host.size() * sizeof(int32_t);
  const VariantBuilder jpeg = [&](const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* pseudo, cudaStream_t st) {
    launch_jpeg_windows(track, d_wins, d_tabs, K, r0, nb, T, H, W, any444, channel_order == LSD_BGR, pseudo, st);
  };
  return score_window_variants(h, "lsd_score_jpeg", "JPEG variants", track, n_frames, H, W, starts_host, audio_starts_host, n_windows, T,
                               mel_full, F, Ta_full, total_v_frames, Ta, K, precision, batch, logits_out, workspace, workspace_bytes,
                               stream, h->variant_tab_host.data(), tab_bytes, tab_bytes, jpeg);
}

// The round-tripped windows themselves, written to a caller buffer by the builder lsd_score_jpeg uses.
extern "C" size_t lsd_jpeg_windows_workspace_bytes(int n_windows, int K, int T, int H, int W) {
  if (n_windows < 1 || K < 1 || K > LSD_MAX_JPEG_VARIANTS || T < 1 || H < 1 || W < 1) return 0;
  return built_windows_workspace_bytes((size_t)K * JPEG_TAB_INTS * sizeof(int32_t), n_windows);
}

extern "C" int lsd_jpeg_windows(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host, int n_windows,
                                int T, const lsd_jpeg* variants, int K, int channel_order, uint8_t* out, void* workspace,
                                size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  bool any444 = false;
  int rc = jpeg_tables_checked(h, "lsd_jpeg_windows", variants, K, channel_order, T, H, W, &any444);
  if (rc) return rc;
  if (n_windows == 0) return LSD_OK;
  if (!track || !starts_host || !out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_jpeg_windows: null pointer argument");
  if (n_windows < 0 || n_frames < 1) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_jpeg_windows: bad extents");
  if ((int64_t)n_windows * K * T > INT32_MAX) return lsd_fail(h, LSD_ERR_SHAPE, "%d windows x %d JPEG variants: too many frames for one call", n_windows, K);
  if ((rc = check_windows(h, starts_host, n_windows, T, n_frames))) return rc;
  const size_t need = lsd_jpeg_windows_workspace_bytes(n_windows, K, T, H, W);
  if (need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  const VariantBuilder jpeg = [&](const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* o, cudaStream_t st) {
    launch_jpeg_windows(track, d_wins, d_tabs, K, r0, nb, T, H, W, any444, channel_order == LSD_BGR, o, st);
  };
  return build_window_variants(h, starts_host, n_windows, K, workspace, stream, h->variant_tab_host.data(),
                               h->variant_tab_host.size() * sizeof(int32_t), out, jpeg);
}

// ------------------------------------------------------------------------------------------------
// Resolution robustness: K down- and re-upscaled copies of every window (resize.cu); tables resize_tables_ints int32
// ------------------------------------------------------------------------------------------------
namespace {
// The checks every resize entry makes before any GPU work; on success h->variant_tab_host holds the K variants' tables.
int resize_tables_checked(lsd_handle* h, const char* fn, const lsd_resize* v, int K, int T, int H, int W) {
  if (!v) return lsd_fail(h, LSD_ERR_ARG, "%s: variants is NULL", fn);
  if (K < 1 || K > LSD_MAX_RESIZE_VARIANTS)
    return lsd_fail(h, LSD_ERR_SHAPE, "K = %d resize variants: expected 1 <= K <= %d", K, LSD_MAX_RESIZE_VARIANTS);
  if (T < 1 || !resize_extents_ok(H, W))
    return lsd_fail(h, LSD_ERR_SHAPE, "%s: bad window extents T=%d H=%d W=%d (frame, face-size frame and tables within shared memory)",
                    fn, T, H, W);
  for (int k = 0; k < K; ++k)
    if (v[k].h < 1 || v[k].h > H || v[k].w < 1 || v[k].w > W)
      return lsd_fail(h, LSD_ERR_SHAPE, "resize variant %d: face size %dx%d is outside 1..%d x 1..%d", k, v[k].h, v[k].w, H, W);
  static_assert(sizeof(lsd_resize) == 2 * sizeof(int32_t), "lsd_resize is two packed int32");
  h->variant_tab_host.resize(resize_tables_ints(K, H, W));
  resize_tables(reinterpret_cast<const int32_t*>(v), K, H, W, h->variant_tab_host.data());
  return 0;
}
}  // namespace

extern "C" size_t lsd_score_resizes_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision) {
  if (batch < 1 || K < 1 || K > LSD_MAX_RESIZE_VARIANTS || !resize_extents_ok(H, W)) return 0;
  return variant_workspace_bytes(h, resize_tables_ints(K, H, W) * sizeof(int32_t), batch, T, H, W, F, Ta, precision);
}

extern "C" int lsd_score_resizes(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                                 const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                                 int total_v_frames, int Ta, const lsd_resize* variants, int K, int precision, int batch,
                                 float* logits_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_score_resizes: no weights loaded");
  const int rc = resize_tables_checked(h, "lsd_score_resizes", variants, K, T, H, W);
  if (rc) return rc;
  const size_t tab_bytes = h->variant_tab_host.size() * sizeof(int32_t);
  const VariantBuilder resize = [&](const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* pseudo, cudaStream_t st) {
    launch_resize_windows(track, d_wins, d_tabs, K, r0, nb, T, H, W, pseudo, st);
  };
  return score_window_variants(h, "lsd_score_resizes", "resize variants", track, n_frames, H, W, starts_host, audio_starts_host, n_windows,
                               T, mel_full, F, Ta_full, total_v_frames, Ta, K, precision, batch, logits_out, workspace, workspace_bytes,
                               stream, h->variant_tab_host.data(), tab_bytes, tab_bytes, resize);
}

// The tap tables of K face sizes, as the kernel reads them: no handle and no device needed.
extern "C" int64_t lsd_resize_tables(const lsd_resize* variants, int K, int H, int W, int32_t* out_or_null) {
  if (!variants) return LSD_ERR_ARG;
  if (K < 1 || K > LSD_MAX_RESIZE_VARIANTS || !resize_extents_ok(H, W)) return LSD_ERR_SHAPE;
  for (int k = 0; k < K; ++k)
    if (variants[k].h < 1 || variants[k].h > H || variants[k].w < 1 || variants[k].w > W) return LSD_ERR_SHAPE;
  if (out_or_null) resize_tables(reinterpret_cast<const int32_t*>(variants), K, H, W, out_or_null);
  return (int64_t)resize_tables_ints(K, H, W);
}

// The resized windows themselves, written to a caller buffer by the builder lsd_score_resizes uses.
extern "C" size_t lsd_resize_windows_workspace_bytes(int n_windows, int K, int T, int H, int W) {
  if (n_windows < 1 || K < 1 || K > LSD_MAX_RESIZE_VARIANTS || T < 1 || !resize_extents_ok(H, W)) return 0;
  return built_windows_workspace_bytes(resize_tables_ints(K, H, W) * sizeof(int32_t), n_windows);
}

extern "C" int lsd_resize_windows(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host, int n_windows,
                                  int T, const lsd_resize* variants, int K, uint8_t* out, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  if (!h) return LSD_ERR_ARG;
  int rc = resize_tables_checked(h, "lsd_resize_windows", variants, K, T, H, W);
  if (rc) return rc;
  if (n_windows == 0) return LSD_OK;
  if (!track || !starts_host || !out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_resize_windows: null pointer argument");
  if (n_windows < 0 || n_frames < 1) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_resize_windows: bad extents");
  if ((int64_t)n_windows * K * T > INT32_MAX)
    return lsd_fail(h, LSD_ERR_SHAPE, "%d windows x %d resize variants: too many frames for one call", n_windows, K);
  if ((rc = check_windows(h, starts_host, n_windows, T, n_frames))) return rc;
  const size_t need = lsd_resize_windows_workspace_bytes(n_windows, K, T, H, W);
  if (need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  const VariantBuilder resize = [&](const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* o, cudaStream_t st) {
    launch_resize_windows(track, d_wins, d_tabs, K, r0, nb, T, H, W, o, st);
  };
  return build_window_variants(h, starts_host, n_windows, K, workspace, stream, h->variant_tab_host.data(),
                               h->variant_tab_host.size() * sizeof(int32_t), out, resize);
}

// ------------------------------------------------------------------------------------------------
// Temporal robustness: K retimed copies of every window (retime.cu); tables K*T lsd_retime entries
// ------------------------------------------------------------------------------------------------
namespace {
// The checks every retime entry makes before any GPU work; on success h->variant_tab_host holds the K*T entries.
int retime_tables_checked(lsd_handle* h, const char* fn, const lsd_retime* v, int K, int T, int H, int W) {
  if (!v) return lsd_fail(h, LSD_ERR_ARG, "%s: variants is NULL", fn);
  if (K < 1 || K > LSD_MAX_RETIMES) return lsd_fail(h, LSD_ERR_SHAPE, "K = %d retime variants: expected 1 <= K <= %d", K, LSD_MAX_RETIMES);
  if (T < 1 || H < 1 || W < 1 || (int64_t)H * W * 3 > INT32_MAX)
    return lsd_fail(h, LSD_ERR_SHAPE, "%s: bad window extents T=%d H=%d W=%d", fn, T, H, W);
  for (int64_t e = 0; e < (int64_t)K * T; ++e) {
    const int k = (int)(e / T), t = (int)(e % T);
    int64_t sum = 0;
    for (int i = 0; i < 4; ++i) {
      if (v[e].src[i] < -T || v[e].src[i] > 2 * T - 1)
        return lsd_fail(h, LSD_ERR_SHAPE, "retime variant %d, frame %d: tap %d src %d is outside %d..%d", k, t, i, v[e].src[i], -T, 2 * T - 1);
      if (v[e].weight[i] < 0)
        return lsd_fail(h, LSD_ERR_ARG, "retime variant %d, frame %d: tap %d has a negative weight %d", k, t, i, v[e].weight[i]);
      sum += v[e].weight[i];
    }
    if (sum != LSD_RETIME_ONE)
      return lsd_fail(h, LSD_ERR_ARG, "retime variant %d, frame %d: weights sum to %lld, not %d", k, t, (long long)sum, LSD_RETIME_ONE);
  }
  static_assert(sizeof(lsd_retime) == 8 * sizeof(int32_t), "lsd_retime is eight packed int32");
  const int32_t* p = reinterpret_cast<const int32_t*>(v);
  h->variant_tab_host.assign(p, p + retime_tables_ints(K, T));
  return 0;
}
}  // namespace

extern "C" size_t lsd_score_retimes_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision) {
  if (batch < 1 || K < 1 || K > LSD_MAX_RETIMES || T < 1) return 0;
  return variant_workspace_bytes(h, retime_tables_ints(K, T) * sizeof(int32_t), batch, T, H, W, F, Ta, precision);
}

extern "C" int lsd_score_retimes(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                                 const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                                 int total_v_frames, int Ta, const lsd_retime* variants, int K, int precision, int batch,
                                 float* logits_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_score_retimes: no weights loaded");
  const int rc = retime_tables_checked(h, "lsd_score_retimes", variants, K, T, H, W);
  if (rc) return rc;
  if ((int64_t)n_windows * K * T > INT32_MAX)
    return lsd_fail(h, LSD_ERR_SHAPE, "%d windows x %d retime variants: too many frames for one call", n_windows, K);
  const size_t tab_bytes = h->variant_tab_host.size() * sizeof(int32_t);
  const VariantBuilder retime = [&](const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* pseudo, cudaStream_t st) {
    launch_retime_windows(track, n_frames, d_wins, d_tabs, K, r0, nb, T, H, W, pseudo, st);
  };
  return score_window_variants(h, "lsd_score_retimes", "retime variants", track, n_frames, H, W, starts_host, audio_starts_host, n_windows,
                               T, mel_full, F, Ta_full, total_v_frames, Ta, K, precision, batch, logits_out, workspace, workspace_bytes,
                               stream, h->variant_tab_host.data(), tab_bytes, tab_bytes, retime);
}

// The retimed windows themselves, written to a caller buffer by the builder lsd_score_retimes uses.
extern "C" size_t lsd_retime_windows_workspace_bytes(int n_windows, int K, int T, int H, int W) {
  if (n_windows < 1 || K < 1 || K > LSD_MAX_RETIMES || T < 1 || H < 1 || W < 1) return 0;
  return built_windows_workspace_bytes(retime_tables_ints(K, T) * sizeof(int32_t), n_windows);
}

extern "C" int lsd_retime_windows(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host, int n_windows,
                                  int T, const lsd_retime* variants, int K, uint8_t* out, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  if (!h) return LSD_ERR_ARG;
  int rc = retime_tables_checked(h, "lsd_retime_windows", variants, K, T, H, W);
  if (rc) return rc;
  if (n_windows == 0) return LSD_OK;
  if (!track || !starts_host || !out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_retime_windows: null pointer argument");
  if (n_windows < 0 || n_frames < 1) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_retime_windows: bad extents");
  if ((int64_t)n_windows * K * T > INT32_MAX)
    return lsd_fail(h, LSD_ERR_SHAPE, "%d windows x %d retime variants: too many frames for one call", n_windows, K);
  if ((rc = check_windows(h, starts_host, n_windows, T, n_frames))) return rc;
  const size_t need = lsd_retime_windows_workspace_bytes(n_windows, K, T, H, W);
  if (need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  const VariantBuilder retime = [&](const int32_t* d_tabs, const int32_t* d_wins, int r0, int nb, uint8_t* o, cudaStream_t st) {
    launch_retime_windows(track, n_frames, d_wins, d_tabs, K, r0, nb, T, H, W, o, st);
  };
  return build_window_variants(h, starts_host, n_windows, K, workspace, stream, h->variant_tab_host.data(),
                               h->variant_tab_host.size() * sizeof(int32_t), out, retime);
}

// ================================================================================================
// Audio variants / offset sweep: K audio windows per video, the video side computed once (bf16_path.cu, VarTail).  Configurations
// the shared route does not cover (fp32, the launch-by-launch token path) run one plain forward / lsd_score_windows per variant.
// ================================================================================================
namespace {
int check_variants(lsd_handle* h, int K) {
  if (K < 1 || K > LSD_MAX_AUDIO_VARIANTS) return lsd_fail(h, LSD_ERR_SHAPE, "K = %d audio variants: expected 1 <= K <= %d", K, LSD_MAX_AUDIO_VARIANTS);
  return 0;
}
bool shared_route(int precision, int T) { return precision == LSD_PREC_BF16 && variants_shared_route(T); }
}  // namespace

extern "C" size_t lsd_forward_audio_variants_workspace_bytes(lsd_handle* h, int B, int K, int T, int H, int W, int F, int Ta, int precision) {
  if (!h || B < 1 || K < 1 || K > LSD_MAX_AUDIO_VARIANTS) return 0;
  if (shared_route(precision, T)) return variants_bf16_bytes(h, B, K, T, H, W, F, Ta);
  const size_t fw = lsd_workspace_bytes(h, B, T, H, W, F, Ta, precision);   // per variant: plain forward + its clips + B logits
  if (fw == 0) return 0;
  return align256(fw) + align256((size_t)B * F * Ta * sizeof(float)) + align256((size_t)B * sizeof(float)) + 256;
}

extern "C" int lsd_forward_audio_variants(lsd_handle* h, const void* video, int video_dtype, int video_layout, const void* audio, int audio_dtype,
                                          int B, int K, int T, int H, int W, int F, int Ta, int precision, float* logits_out,
                                          void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_forward_audio_variants: no weights loaded");
  int rc = check_variants(h, K);
  if (rc) return rc;
  Shapes s;
  if ((rc = make_shapes(h, B, T, H, W, F, Ta, s))) return rc;
  if (B == 0) return LSD_OK;
  if (!video || !audio || !logits_out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_forward_audio_variants: null pointer argument");
  if ((rc = check_dtype(h, video_dtype, "video")) || (rc = check_dtype(h, audio_dtype, "audio"))) return rc;
  if (audio_dtype == LSD_U8) return lsd_fail(h, LSD_ERR_ARG, "audio: uint8 log-mel is not supported");
  if (video_layout != LSD_NCDHW && video_layout != LSD_NDHWC) return lsd_fail(h, LSD_ERR_ARG, "bad video layout %d", video_layout);
  if (precision != LSD_PREC_FP32 && precision != LSD_PREC_BF16) return lsd_fail(h, LSD_ERR_ARG, "bad precision %d", precision);
  const size_t need = lsd_forward_audio_variants_workspace_bytes(h, B, K, T, H, W, F, Ta, precision);
  if (need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = reinterpret_cast<char*>(workspace);
  if (shared_route(precision, T)) {
    if ((rc = forward_variants_bf16(h, B, K, T, H, W, F, Ta, video, video_dtype, video_layout, audio, audio_dtype, logits_out, ws,
                                    workspace_bytes, st))) return rc;
  } else {
    const size_t fw = align256(lsd_workspace_bytes(h, B, T, H, W, F, Ta, precision));
    const size_t clip = (size_t)F * Ta * (audio_dtype == LSD_F32 ? 4 : 2);
    char* aud = ws + fw;
    float* lg = reinterpret_cast<float*>(aud + align256((size_t)B * F * Ta * sizeof(float)));
    for (int k = 0; k < K; ++k) {
      copy_rows_bytes(reinterpret_cast<const char*>(audio) + k * clip, (int64_t)(K * clip), aud, (int64_t)clip, B, (int64_t)clip, st);
      if ((rc = lsd_forward(h, video, video_dtype, video_layout, aud, audio_dtype, B, T, H, W, F, Ta, precision, lg, nullptr, ws, fw, stream)))
        return rc;
      copy_rows_bytes(lg, 4, logits_out + k, (int64_t)K * 4, B, 4, st);
    }
  }
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

extern "C" size_t lsd_score_offsets_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision) {
  if (!h || batch < 1 || K < 1 || K > LSD_MAX_AUDIO_VARIANTS) return 0;
  if (shared_route(precision, T)) {
    const size_t fw = variants_bf16_bytes(h, batch, K, T, H, W, F, Ta);
    if (fw == 0) return 0;
    return align256((size_t)batch * sizeof(int32_t)) + align256((size_t)batch * K * sizeof(int32_t)) + fw + 256;
  }
  const size_t sw = lsd_score_workspace_bytes(h, batch, T, H, W, F, Ta, precision);   // per offset: lsd_score_windows + batch logits
  if (sw == 0) return 0;
  return align256(sw) + align256((size_t)batch * sizeof(float)) + 256;
}

extern "C" int lsd_score_offsets(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                                 const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                                 int total_v_frames, int Ta, const int32_t* offsets_host, int K, int precision, int batch, float* logits_out,
                                 int32_t* eff_audio_starts_host, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_score_offsets: no weights loaded");
  if (!offsets_host) return lsd_fail(h, LSD_ERR_ARG, "lsd_score_offsets: offsets is NULL");
  int rc = check_variants(h, K);
  if (rc) return rc;
  if (n_windows == 0) return LSD_OK;
  if (!track || !starts_host || !mel_full || !logits_out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_score_offsets: null pointer argument");
  if (batch < 1 || n_windows < 0 || n_frames < 1 || Ta_full < 1) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_score_offsets: bad extents");
  if (precision != LSD_PREC_FP32 && precision != LSD_PREC_BF16) return lsd_fail(h, LSD_ERR_ARG, "bad precision %d", precision);
  Shapes s;
  if ((rc = make_shapes(h, batch, T, H, W, F, Ta, s))) return rc;
  for (int i = 0; i < n_windows; ++i)
    if (starts_host[i] < 0 || starts_host[i] + T > n_frames)
      return lsd_fail(h, LSD_ERR_SHAPE, "window %d [%d,%d) is outside the %d-frame track", i, starts_host[i], starts_host[i] + T, n_frames);
  const size_t need = lsd_score_offsets_workspace_bytes(h, batch, K, T, H, W, F, Ta, precision);
  if (need == 0 || need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  // effective start of (i, k): the base start of window i (as lsd_score_windows computes it) moved by offsets[k], clamped the same way
  std::vector<int32_t> eff((size_t)n_windows * K);
  for (int i = 0; i < n_windows; ++i) {
    const long a = base_audio_start(starts_host, audio_starts_host, i, Ta, Ta_full, total_v_frames);
    for (int k = 0; k < K; ++k) eff[(size_t)i * K + k] = (int32_t)clamp_audio_start(a + offsets_host[k], Ta, Ta_full);
  }
  if (eff_audio_starts_host) memcpy(eff_audio_starts_host, eff.data(), eff.size() * sizeof(int32_t));
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = reinterpret_cast<char*>(workspace);
  if (shared_route(precision, T)) {
    const size_t vi = align256((size_t)batch * sizeof(int32_t)), ai = align256((size_t)batch * K * sizeof(int32_t));
    int32_t* d_vs = reinterpret_cast<int32_t*>(ws);
    int32_t* d_as = reinterpret_cast<int32_t*>(ws + vi);
    h->idx_host.resize((size_t)n_windows * (K + 1));   // staged here: the copies below are ordered on the stream
    memcpy(h->idx_host.data(), starts_host, (size_t)n_windows * sizeof(int32_t));
    memcpy(h->idx_host.data() + n_windows, eff.data(), eff.size() * sizeof(int32_t));
    for (int w0 = 0; w0 < n_windows; w0 += batch) {
      const int nb = std::min(batch, n_windows - w0);
      CUDA_OK(h, cudaMemcpyAsync(d_vs, &h->idx_host[w0], nb * sizeof(int32_t), cudaMemcpyHostToDevice, st));
      CUDA_OK(h, cudaMemcpyAsync(d_as, &h->idx_host[n_windows + (size_t)w0 * K], (size_t)nb * K * sizeof(int32_t), cudaMemcpyHostToDevice, st));
      if ((rc = score_offsets_batch_bf16(h, track, n_frames, d_vs, d_as, mel_full, Ta_full, nb, batch, K, T, H, W, F, Ta, logits_out + (size_t)w0 * K,
                                         ws + vi + ai, workspace_bytes - vi - ai, st))) return rc;
    }
  } else {
    const size_t sw = align256(lsd_score_workspace_bytes(h, batch, T, H, W, F, Ta, precision));
    float* lg = reinterpret_cast<float*>(ws + sw);
    std::vector<int32_t> col(batch);
    for (int w0 = 0; w0 < n_windows; w0 += batch) {
      const int nb = std::min(batch, n_windows - w0);
      for (int k = 0; k < K; ++k) {
        for (int i = 0; i < nb; ++i) col[i] = eff[(size_t)(w0 + i) * K + k];
        if ((rc = lsd_score_windows(h, track, n_frames, H, W, starts_host + w0, col.data(), nb, T, mel_full, F, Ta_full, total_v_frames, Ta,
                                    precision, batch, lg, ws, sw, stream))) return rc;
        copy_rows_bytes(lg, 4, logits_out + (size_t)w0 * K + k, (int64_t)K * 4, nb, 4, st);
      }
    }
  }
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

// ================================================================================================
// Audio rows: K device-built (F, Ta) slices per window (occlusion.cu), laid end to end in a pseudo clip and scored as an
// audio-variant sweep with explicit audio starts j*Ta; the clip is never clamped or padded, so the gather copies the slices as built
// ================================================================================================
// Workspace: [variant table | base audio starts of one batch's windows | pseudo clip (F, batch*K*Ta) fp32 | scoring workspace:
// lsd_score_offsets' on the shared route, otherwise lsd_score_windows' at `batch` rows].
namespace {
size_t audio_rows_extra_bytes(size_t table_region, int batch, int K, int F, int Ta) {
  return align256(table_region) + align256((size_t)batch * sizeof(int32_t)) + align256((size_t)F * batch * K * Ta * sizeof(float));
}

size_t audio_rows_workspace_bytes(lsd_handle* h, size_t table_region, int batch, int K, int T, int H, int W, int F, int Ta, int precision) {
  if (!h || batch < 1 || K < 1 || K > LSD_MAX_AUDIO_VARIANTS) return 0;
  const size_t sw = shared_route(precision, T) ? lsd_score_offsets_workspace_bytes(h, batch, K, T, H, W, F, Ta, precision)
                                               : lsd_score_workspace_bytes(h, batch, T, H, W, F, Ta, precision);
  if (sw == 0) return 0;
  return audio_rows_extra_bytes(table_region, batch, K, F, Ta) + align256(sw);
}

// Enqueues on `st` the kernel that writes rows r0 .. r0+nb-1 (window r / K, variant r % K) into columns [j*Ta, (j+1)*Ta) of `clip`,
// j = r - r0; d_tabs: the variant table, d_abase: the base audio starts of windows r0 / K, r0 / K + 1, ...
using AudioRowBuilder = std::function<void(const int32_t* d_tabs, const int32_t* d_abase, int r0, int nb, float* clip, cudaStream_t st)>;

// The common part of lsd_score_audio_occlusions / lsd_score_audio_clips, after each has checked its variants: the remaining argument
// checks, one copy of the variant table (`table_bytes` from tables_host; its region is table_region bytes) and the batch loop.
// `src` is the log-mel the builder reads (checked for NULL), `what` names the variants in messages.
int score_audio_rows(lsd_handle* h, const char* fn, const char* what, const uint8_t* track, int n_frames, int H, int W,
                     const int32_t* starts_host, const int32_t* audio_starts_host, int n_windows, int T, const float* src, int F,
                     int Ta_full, int total_v_frames, int Ta, int K, int precision, int batch, float* logits_out, void* workspace,
                     size_t workspace_bytes, void* stream, const void* tables_host, size_t table_bytes, size_t table_region,
                     const AudioRowBuilder& build) {
  if (n_windows == 0) return LSD_OK;
  if (!track || !starts_host || !src || !logits_out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "%s: null pointer argument", fn);
  if (batch < 1 || n_windows < 0 || n_frames < 1 || Ta_full < 1) return lsd_fail(h, LSD_ERR_SHAPE, "%s: bad extents", fn);
  if ((int64_t)n_windows * K > INT32_MAX || (int64_t)batch * K * Ta > INT32_MAX)
    return lsd_fail(h, LSD_ERR_SHAPE, "%d windows x %d %s in batches of %d: too many rows for one call", n_windows, K, what, batch);
  if (precision != LSD_PREC_FP32 && precision != LSD_PREC_BF16) return lsd_fail(h, LSD_ERR_ARG, "bad precision %d", precision);
  Shapes s;
  int rc = make_shapes(h, batch, T, H, W, F, Ta, s);
  if (rc) return rc;
  if ((rc = check_windows(h, starts_host, n_windows, T, n_frames))) return rc;
  const size_t need = audio_rows_workspace_bytes(h, table_region, batch, K, T, H, W, F, Ta, precision);
  if (need == 0 || need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = reinterpret_cast<char*>(workspace);
  int32_t* d_tabs = reinterpret_cast<int32_t*>(ws);
  int32_t* d_abase = reinterpret_cast<int32_t*>(ws + align256(table_region));
  float* clip = reinterpret_cast<float*>(reinterpret_cast<char*>(d_abase) + align256((size_t)batch * sizeof(int32_t)));
  const size_t extra = audio_rows_extra_bytes(table_region, batch, K, F, Ta);
  char* sws = ws + extra;
  const size_t sws_bytes = workspace_bytes - extra;
  std::vector<int32_t> abase(n_windows), rows((size_t)batch * K);
  for (int i = 0; i < n_windows; ++i) abase[i] = (int32_t)base_audio_start(starts_host, audio_starts_host, i, Ta, Ta_full, total_v_frames);
  for (size_t j = 0; j < rows.size(); ++j) rows[j] = (int32_t)j * Ta;   // row j of a batch: columns [j*Ta, (j+1)*Ta) of the clip
  if (table_bytes) CUDA_OK(h, cudaMemcpyAsync(d_tabs, tables_host, table_bytes, cudaMemcpyHostToDevice, st));
  // One clip serves every batch: batch k+1's builder is enqueued on `st` after every reader of batch k's clip.  On the shared
  // route the only readers are the mel gathers of the audio groups (forward_bf16_impl with a VarTail, not pipelined): group 0 runs
  // on the side stream after ev_start, recorded on `st` behind this batch's builder, and `st` waits for its ev_audio before
  // groups 1.. run on `st` itself, so `st` is past every gather when score_offsets_batch_bf16 returns.  lsd_score_windows
  // gathers the audio of each of its batches on `st`, ahead of the encoders, pipelined or not.
  if (shared_route(precision, T)) {
    const size_t vi = align256((size_t)batch * sizeof(int32_t)), ai = align256((size_t)batch * K * sizeof(int32_t));
    int32_t* d_vs = reinterpret_cast<int32_t*>(sws);
    int32_t* d_as = reinterpret_cast<int32_t*>(sws + vi);
    CUDA_OK(h, cudaMemcpyAsync(d_as, rows.data(), rows.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    for (int w0 = 0; w0 < n_windows; w0 += batch) {
      const int nb = std::min(batch, n_windows - w0);
      CUDA_OK(h, cudaMemcpyAsync(d_vs, starts_host + w0, nb * sizeof(int32_t), cudaMemcpyHostToDevice, st));
      CUDA_OK(h, cudaMemcpyAsync(d_abase, &abase[w0], nb * sizeof(int32_t), cudaMemcpyHostToDevice, st));
      build(d_tabs, d_abase, w0 * K, nb * K, clip, st);
      if ((rc = score_offsets_batch_bf16(h, track, n_frames, d_vs, d_as, clip, nb * K * Ta, nb, batch, K, T, H, W, F, Ta,
                                         logits_out + (size_t)w0 * K, sws + vi + ai, sws_bytes - vi - ai, st))) return rc;
    }
  } else {
    std::vector<int32_t> vrep((size_t)batch * K);   // window i's track start, once per variant
    for (int w0 = 0; w0 < n_windows; w0 += batch) {
      const int nb = std::min(batch, n_windows - w0);
      for (int j = 0; j < nb * K; ++j) vrep[j] = starts_host[w0 + j / K];
      CUDA_OK(h, cudaMemcpyAsync(d_abase, &abase[w0], nb * sizeof(int32_t), cudaMemcpyHostToDevice, st));
      build(d_tabs, d_abase, w0 * K, nb * K, clip, st);
      if ((rc = lsd_score_windows(h, track, n_frames, H, W, vrep.data(), rows.data(), nb * K, T, clip, F, nb * K * Ta, total_v_frames, Ta,
                                  precision, batch, logits_out + (size_t)w0 * K, sws, sws_bytes, stream))) return rc;
    }
  }
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

constexpr size_t AUDIO_OCCLUSION_TABLE_BYTES = (size_t)LSD_MAX_AUDIO_OCCLUSIONS * 4 * sizeof(int32_t);
}  // namespace

// ------------------------------------------------------------------------------------------------
// Audio occlusion evidence: K masked log-mel slices per window (mask_audio_windows_kernel)
// ------------------------------------------------------------------------------------------------
extern "C" size_t lsd_score_audio_occlusions_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision) {
  return audio_rows_workspace_bytes(h, AUDIO_OCCLUSION_TABLE_BYTES, batch, K, T, H, W, F, Ta, precision);
}

extern "C" int lsd_score_audio_occlusions(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                                          const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                                          int total_v_frames, int Ta, const lsd_audio_occlusion* boxes, int K, float fill, int precision,
                                          int batch, float* logits_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_score_audio_occlusions: no weights loaded");
  if (!boxes) return lsd_fail(h, LSD_ERR_ARG, "lsd_score_audio_occlusions: boxes is NULL");
  if (K < 1 || K > LSD_MAX_AUDIO_OCCLUSIONS)
    return lsd_fail(h, LSD_ERR_SHAPE, "K = %d audio occlusion boxes: expected 1 <= K <= %d", K, LSD_MAX_AUDIO_OCCLUSIONS);
  if (!std::isfinite(fill)) return lsd_fail(h, LSD_ERR_ARG, "lsd_score_audio_occlusions: fill %f is not finite", (double)fill);
  for (int k = 0; k < K; ++k) {
    const lsd_audio_occlusion& b = boxes[k];
    if (b.c0 < 0 || b.c0 > b.c1 || b.c1 > Ta || b.f0 < 0 || b.f0 > b.f1 || b.f1 > F)
      return lsd_fail(h, LSD_ERR_SHAPE, "audio box %d [%d,%d)x[%d,%d) is not inside the %d-column x %d-bin window", k, b.c0, b.c1, b.f0,
                      b.f1, Ta, F);
  }
  static_assert(sizeof(lsd_audio_occlusion) == 4 * sizeof(int32_t), "lsd_audio_occlusion is four packed int32");
  const AudioRowBuilder mask = [&](const int32_t* d_boxes, const int32_t* d_abase, int r0, int nb, float* clip, cudaStream_t st) {
    launch_mask_audio_windows(mel_full, F, Ta_full, d_abase, d_boxes, K, r0, nb, Ta, fill, clip, st);
  };
  return score_audio_rows(h, "lsd_score_audio_occlusions", "boxes", track, n_frames, H, W, starts_host, audio_starts_host, n_windows, T,
                          mel_full, F, Ta_full, total_v_frames, Ta, K, precision, batch, logits_out, workspace, workspace_bytes, stream,
                          boxes, (size_t)K * sizeof(lsd_audio_occlusion), AUDIO_OCCLUSION_TABLE_BYTES, mask);
}

// ------------------------------------------------------------------------------------------------
// Audio robustness: K degraded copies of one clip (audio_degrade.cu), and every window scored against K clip log-mels
// ------------------------------------------------------------------------------------------------
// Degrade workspace: [variant table, band taps, impulse responses (at most K * DEGRADE_MAX_RIR floats) | noise partial sums |
// band intermediate K * ceil(n / 2) floats]
namespace {
size_t degrade_table_region(int K) { return ((size_t)K * DEGRADE_TAB_INTS + 2 * (41 + 81) + (size_t)K * DEGRADE_MAX_RIR) * sizeof(int32_t); }
}  // namespace

extern "C" size_t lsd_degrade_audio_workspace_bytes(int64_t n, int K) {
  if (n < 1 || K < 1 || K > LSD_MAX_AUDIO_DEGRADATIONS) return 0;
  return align256(degrade_table_region(K)) + align256(degrade_partials_bytes(K)) + align256((size_t)K * ((n + 1) / 2) * sizeof(float));
}

extern "C" int lsd_degrade_audio(lsd_handle* h, const float* pcm, int64_t n, const lsd_audio_degradation* variants, int K, float* out,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (K < 1 || K > LSD_MAX_AUDIO_DEGRADATIONS)
    return lsd_fail(h, LSD_ERR_SHAPE, "K = %d audio degradations: expected 1 <= K <= %d", K, LSD_MAX_AUDIO_DEGRADATIONS);
  if (n < 1) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_degrade_audio: %lld samples, expected at least 1", (long long)n);
  if ((int64_t)K * n > INT64_MAX / 8) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_degrade_audio: %d x %lld samples is too large", K, (long long)n);
  if (!pcm || !variants || !out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_degrade_audio: null pointer argument");
  const int all = LSD_AD_REVERB | LSD_AD_NOISE | LSD_AD_CLIP | LSD_AD_BAND | LSD_AD_MULAW;
  for (int k = 0; k < K; ++k) {
    const lsd_audio_degradation& v = variants[k];
    if (v.stages & ~all) return lsd_fail(h, LSD_ERR_ARG, "audio degradation %d: unknown stage bits 0x%x", k, v.stages & ~all);
    if ((v.stages & LSD_AD_REVERB) && !(std::isfinite(v.rt60) && v.rt60 >= 0.05f && v.rt60 <= 2.0f))
      return lsd_fail(h, LSD_ERR_ARG, "audio degradation %d: rt60 %g s is outside [0.05, 2]", k, (double)v.rt60);
    if ((v.stages & LSD_AD_NOISE) && !(std::isfinite(v.snr_db) && v.snr_db >= -20.f && v.snr_db <= 60.f))
      return lsd_fail(h, LSD_ERR_ARG, "audio degradation %d: snr %g dB is outside [-20, 60]", k, (double)v.snr_db);
    if ((v.stages & LSD_AD_CLIP) && !(std::isfinite(v.gain_db) && v.gain_db >= 0.f && v.gain_db <= 40.f))
      return lsd_fail(h, LSD_ERR_ARG, "audio degradation %d: gain %g dB is outside [0, 40]", k, (double)v.gain_db);
    if ((v.stages & LSD_AD_BAND) && v.band_rate != 8000 && v.band_rate != 4000)
      return lsd_fail(h, LSD_ERR_ARG, "audio degradation %d: band_rate %d is not 8000 or 4000", k, v.band_rate);
  }
  const size_t need = lsd_degrade_audio_workspace_bytes(n, K);
  if (need > workspace_bytes) return lsd_fail(h, LSD_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  degrade_tables(variants, K, h->variant_tab_host);   // kept until the next call: the copy below is asynchronous
  char* ws = reinterpret_cast<char*>(workspace);
  int32_t* d_tab = reinterpret_cast<int32_t*>(ws);
  double* part = reinterpret_cast<double*>(ws + align256(degrade_table_region(K)));
  float* mid = reinterpret_cast<float*>(reinterpret_cast<char*>(part) + align256(degrade_partials_bytes(K)));
  CUDA_OK(h, cudaMemcpyAsync(d_tab, h->variant_tab_host.data(), h->variant_tab_host.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  launch_degrade_audio(pcm, n, variants, K, d_tab, part, mid, out, st);
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

extern "C" size_t lsd_score_audio_clips_workspace_bytes(lsd_handle* h, int batch, int K, int T, int H, int W, int F, int Ta, int precision) {
  return audio_rows_workspace_bytes(h, 0, batch, K, T, H, W, F, Ta, precision);
}

extern "C" int lsd_score_audio_clips(lsd_handle* h, const uint8_t* track, int n_frames, int H, int W, const int32_t* starts_host,
                                     const int32_t* audio_starts_host, int n_windows, int T, const float* mels, int F, int Ta_full,
                                     int total_v_frames, int Ta, int K, int precision, int batch, float* logits_out, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_score_audio_clips: no weights loaded");
  if (K < 1 || K > LSD_MAX_AUDIO_DEGRADATIONS)
    return lsd_fail(h, LSD_ERR_SHAPE, "K = %d clips: expected 1 <= K <= %d", K, LSD_MAX_AUDIO_DEGRADATIONS);
  const AudioRowBuilder gather = [&](const int32_t*, const int32_t* d_abase, int r0, int nb, float* clip, cudaStream_t st) {
    launch_gather_audio_variants(mels, F, Ta_full, d_abase, K, r0, nb, Ta, clip, st);
  };
  return score_audio_rows(h, "lsd_score_audio_clips", "clips", track, n_frames, H, W, starts_host, audio_starts_host, n_windows, T, mels, F,
                          Ta_full, total_v_frames, Ta, K, precision, batch, logits_out, workspace, workspace_bytes, stream, nullptr, 0, 0,
                          gather);
}

// ================================================================================================
// Sub-paths (tensor-core route): AudioEncoder.forward and CrossModalAttention + TemporalTransformer
// ================================================================================================
extern "C" size_t lsd_audio_encoder_workspace_bytes(lsd_handle* h, int B, int F, int Ta) {
  return h ? audio_encoder_bf16_bytes(h, B, F, Ta) : 0;
}
// dst[i] = fl(src[i] / 255.0f): IEEE division, the reference's own operation (video.py:552-556); 16 values per thread
__global__ void expand_u8_kernel(const uint4* __restrict__ src, float4* __restrict__ dst, int64_t n16) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n16) return;
  const uint4 v = src[i];
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int q = 0; q < 4; ++q)
    dst[4 * i + q] = make_float4(__fdiv_rn((float)(w[q] & 0xffu), 255.0f), __fdiv_rn((float)((w[q] >> 8) & 0xffu), 255.0f),
                                 __fdiv_rn((float)((w[q] >> 16) & 0xffu), 255.0f), __fdiv_rn((float)(w[q] >> 24), 255.0f));
}
extern "C" int lsd_expand_u8(const uint8_t* src, float* dst, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && (!src || !dst)) || (n & 15) || (reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(dst) & 15)) return LSD_ERR_ARG;
  if (n == 0) return LSD_OK;
  const int64_t n16 = n / 16;
  expand_u8_kernel<<<(unsigned)((n16 + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint4*>(src), reinterpret_cast<float4*>(dst), n16);
  lsd::count_launch();
  return cudaGetLastError() == cudaSuccess ? LSD_OK : LSD_ERR_CUDA;
}

extern "C" int lsd_audio_encoder(lsd_handle* h, const void* audio, int audio_dtype, int B, int F, int Ta, float* feats_out,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_audio_encoder: no weights loaded");
  if (B < 0 || F < 1 || Ta < 1) return lsd_fail(h, LSD_ERR_SHAPE, "expected audio (B,1,F,T_a) with positive extents, got B=%d F=%d Ta=%d", B, F, Ta);
  if (B == 0) return LSD_OK;
  if (!audio || !feats_out || !workspace) return lsd_fail(h, LSD_ERR_ARG, "lsd_audio_encoder: null pointer argument");
  int rc = check_dtype(h, audio_dtype, "audio");
  if (rc) return rc;
  if (audio_dtype == LSD_U8) return lsd_fail(h, LSD_ERR_ARG, "audio: uint8 log-mel is not supported");
  ENTER_DEVICE(h);
  rc = audio_encoder_bf16_run(h, B, F, Ta, audio, audio_dtype, feats_out, reinterpret_cast<char*>(workspace), workspace_bytes,
                              reinterpret_cast<cudaStream_t>(stream));
  if (rc) return rc;
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}
extern "C" size_t lsd_token_path_workspace_bytes(lsd_handle* h, int B, int T, int Ta_tokens) {
  return h ? token_path_bf16_bytes(h, B, T, Ta_tokens) : 0;
}
extern "C" int lsd_token_path(lsd_handle* h, const float* v_emb, const float* a_emb, int B, int T, int Ta_tokens, float* fused_out,
                              float* cls_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (!h->loaded) return lsd_fail(h, LSD_ERR_WEIGHTS, "lsd_token_path: no weights loaded");
  if (B < 0 || T < 1 || Ta_tokens < 1) return lsd_fail(h, LSD_ERR_SHAPE, "expected v_emb (B,T,256) and a_emb (B,T_a,256), got B=%d T=%d T_a=%d", B, T, Ta_tokens);
  if (B == 0) return LSD_OK;
  if (!v_emb || !a_emb || !workspace || (!fused_out && !cls_out)) return lsd_fail(h, LSD_ERR_ARG, "lsd_token_path: null pointer argument");
  ENTER_DEVICE(h);
  int rc = token_path_bf16_run(h, B, T, Ta_tokens, v_emb, a_emb, fused_out, cls_out, reinterpret_cast<char*>(workspace), workspace_bytes,
                               reinterpret_cast<cudaStream_t>(stream));
  if (rc) return rc;
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

// ================================================================================================
// Speaking alignment / mouth motion statistics (host numpy loops of predictor.py:333-419, per window)
// ================================================================================================
extern "C" int lsd_track_motion(lsd_handle* h, const void* video, int dtype, int layout, int n_frames, int H, int W,
                                float* motion_full, float* motion_low, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (n_frames < 1 || H < 2 || W < 1) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_track_motion: bad extents n_frames=%d H=%d W=%d", n_frames, H, W);
  if (n_frames < 2) return LSD_OK;
  if (!video || !motion_full || !motion_low) return lsd_fail(h, LSD_ERR_ARG, "lsd_track_motion: null pointer argument");
  if (!((dtype == LSD_U8 && layout == LSD_NDHWC) || (dtype == LSD_F32 && layout == LSD_NCDHW)))
    return lsd_fail(h, LSD_ERR_ARG, "lsd_track_motion: supported inputs are a uint8 (n,H,W,3) track or a float32 (3,T,H,W) window");
  ENTER_DEVICE(h);
  lsd::launch_track_motion(video, layout == LSD_NDHWC ? 1 : 0, n_frames, H, W, motion_full, motion_low, reinterpret_cast<cudaStream_t>(stream));
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

extern "C" int lsd_speech_stats(lsd_handle* h, const float* motion_full, const float* motion_low, int n_frames, const int32_t* starts_host,
                                const int32_t* audio_starts_host, int n_windows, int T, const float* mel_full, int F, int Ta_full,
                                int total_v_frames, int Ta, float* speaking_out, float* mouth_motion_out, float* audio_energy_out,
                                int32_t* idx_scratch, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (n_windows == 0) return LSD_OK;
  if (!motion_full || !motion_low || !starts_host || !mel_full || !speaking_out || !mouth_motion_out || !audio_energy_out || !idx_scratch)
    return lsd_fail(h, LSD_ERR_ARG, "lsd_speech_stats: null pointer argument");
  if (n_windows < 0 || T < 1 || Ta < 1 || F < 1 || Ta_full < 1 || T > lsd::speech_stats_max() || Ta > lsd::speech_stats_max())
    return lsd_fail(h, LSD_ERR_SHAPE, "lsd_speech_stats: bad extents (T and Ta must be in [1, %d])", lsd::speech_stats_max());
  for (int i = 0; i < n_windows; ++i)
    if (starts_host[i] < 0 || starts_host[i] + T > n_frames)
      return lsd_fail(h, LSD_ERR_SHAPE, "window %d [%d,%d) is outside the %d-frame track", i, starts_host[i], starts_host[i] + T, n_frames);
  ENTER_DEVICE(h);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  h->idx_host.resize((size_t)2 * n_windows);
  for (int i = 0; i < n_windows; ++i) {
    h->idx_host[i] = starts_host[i];
    h->idx_host[n_windows + i] = (int32_t)base_audio_start(starts_host, audio_starts_host, i, Ta, Ta_full, total_v_frames);   // predictor.py:540-547
  }
  CUDA_OK(h, cudaMemcpyAsync(idx_scratch, h->idx_host.data(), (size_t)2 * n_windows * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  lsd::launch_speech_stats(motion_full, motion_low, idx_scratch, idx_scratch + n_windows, n_windows, T, mel_full, F, Ta_full, Ta, speaking_out,
                           mouth_motion_out, audio_energy_out, st);
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

// ================================================================================================
// Energy VAD (detect_voice_activity, app/preprocessing/audio.py:178-230)
// ================================================================================================
extern "C" int lsd_vad_frames(int64_t n_samples) { return n_samples <= 0 ? 0 : (int)((n_samples + 159) / 160); }
extern "C" int lsd_frame_energy(lsd_handle* h, const float* pcm, int64_t n_samples, float* energy_out, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (n_samples < 0) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_frame_energy: negative length");
  if (n_samples == 0) return LSD_OK;
  if (!pcm || !energy_out) return lsd_fail(h, LSD_ERR_ARG, "lsd_frame_energy: null pointer argument");
  ENTER_DEVICE(h);
  lsd::launch_frame_energy(pcm, n_samples, lsd_vad_frames(n_samples), energy_out, reinterpret_cast<cudaStream_t>(stream));
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}
extern "C" int lsd_vad_mask(lsd_handle* h, const float* energy, int n_frames, float threshold, uint8_t* mask_out, void* stream) {
  if (!h) return LSD_ERR_ARG;
  if (n_frames < 0) return lsd_fail(h, LSD_ERR_SHAPE, "lsd_vad_mask: negative length");
  if (n_frames == 0) return LSD_OK;
  if (!energy || !mask_out) return lsd_fail(h, LSD_ERR_ARG, "lsd_vad_mask: null pointer argument");
  ENTER_DEVICE(h);
  lsd::launch_vad_mask(energy, n_frames, threshold, mask_out, reinterpret_cast<cudaStream_t>(stream));
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

// ================================================================================================
// Introspection
// ================================================================================================
extern "C" int lsd_planar_stage_read(lsd_handle* h, const char* name, const char* name_lo_or_null, const void* workspace, float* out,
                                     int64_t out_elems, int H_full, int W_full, void* stream) {
  if (!h || !name || !workspace || !out) return lsd_fail(h, LSD_ERR_ARG, "lsd_planar_stage_read: null argument");
  ENTER_DEVICE(h);
  int rc = planar_stage_read(h, name, name_lo_or_null, reinterpret_cast<const char*>(workspace), out, out_elems, H_full, W_full,
                             reinterpret_cast<cudaStream_t>(stream));
  if (rc) return rc;
  CUDA_OK(h, cudaGetLastError());
  return LSD_OK;
}

extern "C" int64_t lsd_state_generation(lsd_handle* h) { return h ? h->generation : -1; }

extern "C" int lsd_workspace_invalidate(lsd_handle* h) {
  if (!h) return LSD_ERR_ARG;
  for (WsSig& w : h->ws_sig) w.ptr = nullptr;
  return LSD_OK;
}

extern "C" int lsd_profile_enable(lsd_handle* h, int on) {
  if (!h) return LSD_ERR_ARG;
  h->prof.want = on;   // 1: fp32 conv kernel class, 2: tcgen05 conv kernel class
  h->prof.on = false;
  h->prof.used = 0; h->prof.flops = 0; h->prof.launches = 0;
  return LSD_OK;
}
extern "C" int lsd_profile_get(lsd_handle* h, double* kernel_ms, int64_t* launches, double* flops) {
  if (!h) return LSD_ERR_ARG;
  double ms = 0;
  for (size_t i = 0; i + 1 < h->prof.used; i += 2) {
    cudaError_t e = cudaEventSynchronize(h->prof.ev[i + 1]);
    float t = 0;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&t, h->prof.ev[i], h->prof.ev[i + 1]);
    if (e != cudaSuccess) return lsd_fail(h, LSD_ERR_CUDA, "lsd_profile_get: %s", cudaGetErrorString(e));
    ms += t;
  }
  if (kernel_ms) *kernel_ms = ms;
  if (launches) *launches = h->prof.launches;
  if (flops) *flops = h->prof.flops;
  h->prof.used = 0; h->prof.flops = 0; h->prof.launches = 0;
  return LSD_OK;
}
extern "C" int lsd_stage_count(lsd_handle* h) { return h ? (int)h->stages.size() : 0; }
extern "C" const char* lsd_stage_name(lsd_handle* h, int i) {
  if (!h || i < 0 || i >= (int)h->stages.size()) return nullptr;
  return h->stages[i].name.c_str();
}
extern "C" int lsd_stage_info(lsd_handle* h, const char* name, size_t* offset_bytes, int64_t* numel, int* dtype) {
  if (!h || !name) return LSD_ERR_ARG;
  for (const Stage& s : h->stages)
    if (s.name == name) {
      if (offset_bytes) *offset_bytes = s.offset;
      if (numel) *numel = s.numel;
      if (dtype) *dtype = s.dtype;
      return LSD_OK;
    }
  return lsd_fail(h, LSD_ERR_ARG, "unknown stage %s", name);
}
