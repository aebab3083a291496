// Internal host-side state shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <unordered_map>
#include <string>
#include <vector>

struct ConvP {            // one folded conv / linear in the fp32 device arena (offsets in floats)
  size_t w_off = 0, scale_off = 0, shift_off = 0;
  bool has_scale = false;
  int Cin = 0, Cout = 0, kt = 1, kh = 1, kw = 1;
};

struct Stage {            // named intermediate of the last forward (byte offset into the caller's workspace)
  std::string name;
  size_t offset = 0;
  int64_t numel = 0;
  int dtype = 0;
};

struct BTap { int orig, dt, dh, dw; };                       // original tap index + input shift (in the band's plane set)
struct BBand { int set; std::vector<BTap> taps; };
struct BGroup { std::vector<BBand> bands; int Cin = 0, taps_total = 0, k16 = 0, toeplitz = 0, src = 0; size_t w_off = 0, slice_stride = 0; };  // src: 0 main input, 1 downsample input, 2 low part of the main input  // w_off: bf16 elements into barena
struct BLayer { std::vector<BGroup> groups; int Cout = 0, ntile = 0; size_t bias_off = 0; bool halves = false; };  // halves: weights packed as two ntile/2-column slices (CTA pairs)            // bias_off: floats into bbias

struct Prof {             // CUDA-event brackets around the dominant kernel class (lsd_profile_*)
  int want = 0;           // 0 off, 1 fp32 conv kernel, 2 tcgen05 conv kernel
  bool on = false;
  std::vector<cudaEvent_t> ev;
  size_t used = 0;
  double flops = 0;
  int64_t launches = 0;
  void begin(cudaStream_t st, double fl, int cls = 1) {
    on = (want == cls);
    if (!on) return;
    while (ev.size() < used + 2) { cudaEvent_t e; cudaEventCreate(&e); ev.push_back(e); }
    cudaEventRecord(ev[used], st);
    flops += fl; ++launches;
  }
  void end(cudaStream_t st) {
    if (!on) return;
    cudaEventRecord(ev[used + 1], st);
    used += 2;
  }
};

// Layout of a planar bf16 buffer: plain (one plane set, the map itself), parity-split (4 half-resolution plane sets by (h&1, w&1),
// or by h&1 only for the stride-(2,1) audio layers: sets 0 and 2), folded (one plane set per map position, frame-row geometry),
// or bf16 pixel rows (stem / laplacian / audio stem inputs: 2 h-parity sets of 2-pixel units, not a channel map).
enum PlanarKind { PK_PLAIN = 0, PK_PARITY_H = 1, PK_PARITY_HW = 2, PK_FOLD = 3, PK_ROWS = 4 };

struct PlanarStage {      // planar bf16 buffer of the last tensor-core forward (introspection: lsd_planar_stage_read)
  size_t off = 0;
  int C = 0, sets = 1;
  int kind = PK_PLAIN;
  int map_h = 0, map_w = 0;   // full-resolution extent of the map the buffer holds
  int64_t plane_stride = 0, set_stride = 0, origin = 0;
  int N = 0, T = 0, H = 0, W = 0, ot = 0, oh = 0, hp_extra = 0, ow = 0, wp_extra = 0;
};

struct WsSig { const void* ptr = nullptr; size_t bytes = 0; int shape[6] = {0, 0, 0, 0, 0, 0}; };

struct lsd_handle {
  int device = 0;
  int num_sms = 148;
  std::string err;
  bool loaded = false;
  float* warena = nullptr;                 // fp32 packed weights
  float lapw_host[81] = {0};               // host copy of the 3->3 laplacian conv weights [tap][ci][co]: passed to video_rows by value
  void* barena = nullptr;                  // bf16 UMMA-packed weights
  std::map<std::string, ConvP> convs;
  std::map<std::string, size_t> vecs;      // small fp32 vectors (offsets into warena)
  float* bbias = nullptr;                  // fp32 biases of the bf16 layers
  // fused temporal-transformer kernel (tok_fused.cu): fp16 weight stream, per-layer stage sizes, small fp32 vectors
  void* tokfr_w = nullptr;                 // fused token-path front (tok_front.cu): packed fp16 weight stream + fp32 vectors
  float* tokfr_vec = nullptr;
  void* tokf_w = nullptr;
  uint32_t* tokf_stage_bytes = nullptr;
  float* tokf_vec = nullptr;
  int tokf_n_stage = 0;
  uint32_t tokf_layer_bytes = 0;
  std::map<std::string, BLayer> blayers;
  WsSig ws_sig[3];                         // bf16 workspaces whose zero padding is initialised (see ws_prepare in bf16_path.cu)
  // cross-batch pipelining of lsd_score_windows: the tail of batch k (audio encoder, token path, head; artifact branch on the
  // side stream) runs on tail_stream while the main stream already runs the visual encoder of batch k+1
  cudaStream_t tail_stream = nullptr;
  cudaEvent_t ev_front[2] = {nullptr, nullptr}, ev_tail_done[2] = {nullptr, nullptr};
  std::vector<Stage> stages;
  std::map<std::string, PlanarStage> planar_stages;
  std::vector<int32_t> idx_host;
  std::vector<int32_t> variant_tab_host;   // lsd_score_warps / lsd_score_jpeg / lsd_score_resizes / lsd_score_retimes: host copy of the variant tables, kept until the next call (async copy)
  Prof prof;
  cudaStream_t side_stream = nullptr;      // artifact branch runs here, concurrently with the token path
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_start = nullptr, ev_audio = nullptr;
  cudaStream_t side2_stream = nullptr;     // high-frequency branch, next to the temporal-inconsistency convolutions on side_stream
  cudaEvent_t ev_join2 = nullptr;
  // independent pieces of the token path (the two attention directions, the three multi-scale branches) run side by side
  cudaStream_t tok_stream[2] = {nullptr, nullptr};
  cudaEvent_t ev_tok_fork = nullptr, ev_tok_join[2] = {nullptr, nullptr};
  int64_t launches0 = 0;
  int64_t generation = 0;                  // bumped whenever device addresses baked into earlier launches become stale (see lsd_state_generation)
  // stage programs of the tcgen05 launches (umma_conv.cuh): built on the host once per (layer, shapes, workspace), cached here
  char* prog_arena = nullptr;
  size_t prog_cap = 0, prog_cursor = 0;
  std::unordered_map<uint64_t, const void*> prog_cache;
  // temporal-ring stem (stem_ring.cu): packed N = 192 weights inside barena, step tables per (batch, frames, geometry)
  size_t stem_ring_w_off = 0;              // bf16 elements into barena; 0 = not packed
  struct RingTab { void* dev = nullptr; int nsteps = 0, grid = 0; };
  std::unordered_map<uint64_t, RingTab> ring_tabs;
  // log-mel tables (device): hann[400], cos[400], sin[400], melw[80*32], lo[80], cnt[80]
  void* mel_tables = nullptr;
  const float *d_hann = nullptr, *d_cos = nullptr, *d_sin = nullptr, *d_melw = nullptr;
  const int *d_mel_lo = nullptr, *d_mel_cnt = nullptr;
  const void* d_w400 = nullptr;            // float2[400]: exp(-2*pi*i*m/400)
  void* lm_clips = nullptr;                // device clip table of the batched log-mel kernel (grows on demand)
  size_t lm_clips_cap = 0;
  std::vector<char> lm_clips_host;
  cudaEvent_t ev_lm_clips = nullptr;       // recorded after the kernels that read lm_clips; the next upload waits on it
  bool lm_clips_used = false;
};

int lsd_fail(lsd_handle* h, int code, const char* fmt, ...);
int init_logmel_tables(lsd_handle* h);

// bf16 tensor-core path (bf16_path.cu)
int pack_bf16_weights(lsd_handle* h, const std::vector<float>& f32_arena);
void make_plan_bf16(lsd_handle* h, int B, int T, int H, int W, int F, int Ta, std::vector<Stage>& stages, size_t& bytes);
#include "../../include/lsd_b200.h"
int forward_bf16(lsd_handle* h, int B, int T, int H, int W, int F, int Ta, const void* video, int vdt, int vlayout,
                 const void* audio, int adt, float* logits, const lsd_aux* aux, char* ws, size_t ws_bytes,
                 cudaStream_t st, bool inputs_ready);
size_t audio_encoder_bf16_bytes(lsd_handle* h, int B, int F, int Ta);
int audio_encoder_bf16_run(lsd_handle* h, int B, int F, int Ta, const void* audio, int adt, float* feats_out, char* ws, size_t ws_bytes,
                           cudaStream_t st);
size_t token_path_bf16_bytes(lsd_handle* h, int B, int T, int TA);
int token_path_bf16_run(lsd_handle* h, int B, int T, int TA, const float* v_emb, const float* a_emb, float* fused_out, float* cls_out,
                        char* ws, size_t ws_bytes, cudaStream_t st);
int score_batch_bf16(lsd_handle* h, const uint8_t* track, int n_frames, const int32_t* d_vstarts, const int32_t* d_astarts,
                     const float* mel_full, int Ta_full, int nb, int T, int H, int W, int F, int Ta, float* logits,
                     char* ws, size_t ws_bytes, cudaStream_t st, int pipe_parity = -1, float* feats_out = nullptr);
int ensure_pipeline(lsd_handle* h);
// shared-visual forward: K audio windows per video, visual front once (bf16_path.cu, VarTail)
bool variants_shared_route(int T);
size_t variants_bf16_bytes(lsd_handle* h, int B, int K, int T, int H, int W, int F, int Ta);
int forward_variants_bf16(lsd_handle* h, int B, int K, int T, int H, int W, int F, int Ta, const void* video, int vdt, int vlayout,
                          const void* audio, int adt, float* logits, char* ws, size_t ws_bytes, cudaStream_t st);
int score_offsets_batch_bf16(lsd_handle* h, const uint8_t* track, int n_frames, const int32_t* d_vstarts, const int32_t* d_astarts,
                             const float* mel_full, int Ta_full, int nb, int batch, int K, int T, int H, int W, int F, int Ta, float* logits,
                             char* ws, size_t ws_bytes, cudaStream_t st);
int planar_stage_read(lsd_handle* h, const char* name, const char* name_lo, const char* ws, float* out, int64_t out_elems, int Hf, int Wf,
                      cudaStream_t st);
