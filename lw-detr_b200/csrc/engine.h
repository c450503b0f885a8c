// LW-DETR forward engine: weight packing (folding, layout changes, 16-bit conversion) and the fixed
// kernel schedule for one (batch size, input resolution).  Host-only interface; see engine.cpp.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <functional>
#include <map>
#include <string>
#include <vector>

#include "lwdetr_b200.h"

namespace lwb {

struct HostTensor {
  const float* data;
  long long numel;
};

struct Capture {
  std::string label;
  float* dst;
  long long capacity;   // in floats
  long long written;    // rows*cols actually written (or -1 if label not found)
};

struct Op {
  std::string label;
  std::function<int(cudaStream_t)> run;
  // output description for debug captures
  const void* out = nullptr;
  long long rows = 0;
  int cols = 0, ld = 0, fp32 = 0;
  double flops = 0, bytes = 0;
  bool reads_input = false;   // consumes caller-owned pointers (images, mask): launched eagerly, never captured in the graph
};

// One forward's input: the image batch in one of four encodings plus the optional NestedTensor padding mask.
enum : int { IN_F32_NCHW = 0, IN_16_NCHW = 1, IN_U8_NHWC = 2, IN_U8_FRAMES = 3 };
struct ForwardIn {
  const void* images = nullptr;   // DEVICE [B,3,R,R] fp32 / compute dtype, or [B,R,R,3] uint8
  int kind = IN_F32_NCHW;
  const lwdetr_frame* frames = nullptr;   // IN_U8_FRAMES: HOST [B] descriptors of uint8 frames of any size (resized to R)
  const uint8_t* mask = nullptr;  // DEVICE bool [B,R,R] (True = padded pixel) or null
  float mean[3] = {0.f, 0.f, 0.f}, stdv[3] = {1.f, 1.f, 1.f};   // IN_U8_NHWC / IN_U8_FRAMES: (x/255 - mean) / std
};

class Engine {
 public:
  Engine(const lwdetr_config& cfg, int dtype);
  ~Engine();
  int load_weights(const std::map<std::string, HostTensor>& w, std::string* err);
  // R: input side in pixels (a multiple of 64; the caller checks the supported range)
  int forward(const ForwardIn& in, int B, int R, float* pred_logits, float* pred_boxes,
              const lwdetr_aux_out* aux, const int32_t* topk_override, cudaStream_t st, std::string* err);
  // Forget the schedule (and the position table it built): the next forward re-plans from the current arena.
  void invalidate_plan() { drop_graphs(); planned_B_ = 0; }
  void add_capture(const char* label, float* dst, long long cap) { captures_.push_back({label, dst, cap, -1}); }
  void clear_captures() { captures_.clear(); }
  long long capture_written(int i) const { return i < (int)captures_.size() ? captures_[i].written : -1; }
  int set_option(const char* name, int value);
  // packed weight arena (device): base pointer and bytes in use - identical layout on every rank with the same config / dtype
  void* arena_ptr() const { return warena_.p; }
  size_t arena_used() const { return woff_; }
  bool weights_loaded() const { return weights_loaded_; }
  int device() const { return device_; }
  int num_ops() const { return static_cast<int>(ops_.size()); }
  const Op& op(int i) const { return ops_[i]; }
  const lwdetr_config& config() const { return cfg_; }
  // per-op timing of the last planned batch (CUDA events, `iters` runs per op); returns ms per op
  int profile_ops(int iters, std::vector<float>* ms, cudaStream_t st, std::string* err);

 private:
  struct DevBuf { void* p = nullptr; size_t bytes = 0; };
  int plan(int B, int R, std::string* err);
  void* walloc(size_t bytes);      // weight arena (bump)
  void* salloc(size_t bytes);      // workspace arena (bump)
  std::vector<uint16_t> to16(const std::vector<float>& v) const;   // round to the compute dtype
  void* upload16(const std::vector<float>& v);
  // ViT position table of a G x G token grid -> dst (DEVICE, compute dtype, [G*G, C] in the window-major row order of the
  // patch-embedding GEMM), built from the raw 14 x 14 table kept in the weight arena ("pos_raw").  Synchronous.
  int upload_pos_table(int G, void* dst);
  float* upload32(const std::vector<float>& v);
  int do_capture(const Op& op, cudaStream_t st);

  lwdetr_config cfg_;
  int dtype_;
  int device_ = 0;    // CUDA device the engine was created on; every entry point switches to it (one handle per device)
  int planned_B_ = 0, planned_R_ = 0;
  bool weights_loaded_ = false;
  int use_graph_ = 0;
  int fuse_ln_ = 1;   // ViT LayerNorms folded into the consuming GEMM's epilogue (option "fuse_layernorm")
  // CUDA graphs: the two ops that read caller-owned memory (mask tables, patch gather) are launched eagerly on the
  // caller's stream; everything behind them only touches engine-owned buffers and is ONE executable graph per planned
  // batch size - whatever tensor, input encoding or mask the caller passes.  (The test-only top-k override pointer is
  // the one caller pointer left inside, hence the key.)  Captured on an internal stream: the caller's stream may be the
  // legacy default stream, which cannot be captured.
  struct GraphKey { const void* topk; bool operator<(const GraphKey& o) const { return topk < o.topk; } };
  std::map<GraphKey, cudaGraphExec_t> graphs_;
  cudaStream_t gstream_ = nullptr;
  cudaEvent_t ev_in_ = nullptr, ev_out_ = nullptr;
  int eager_runs_ = 0;
  void drop_graphs();
  std::vector<Op> ops_;
  std::vector<Capture> captures_;
  // arenas
  DevBuf warena_, sarena_;
  size_t woff_ = 0, soff_ = 0;
  // packed weights (device pointers), keyed by short names
  std::map<std::string, void*> W_;
  std::map<std::string, float*> F_;
  std::vector<uint8_t> invalid_rows_;   // per memory token
  // live I/O pointers patched into the schedule at forward() time
  ForwardIn in_;
  std::vector<lwdetr_frame> frames_;   // IN_U8_FRAMES: the last forward's descriptors (profile_ops re-runs them)
  int patch_op_ = -1;                  // index of the input-reading "patch_gather" op in ops_
  double patch_bytes_ = 0;             // its bytes for a [B,3,R,R] input; a frames forward reports the frames' bytes
  const int32_t* in_topk_override_ = nullptr;
  // result buffers (engine owned)
  float* out_logits_ = nullptr;   // [layers, B, nq, ldc_]
  int ldc_ = 96;                  // row pitch of the class-logit buffers: num_classes rounded up to 32
  float* out_boxes_ = nullptr;    // [layers, B, nq, 4]
  float* out_enc_logits_ = nullptr;  // [B, nq, ncls]
  float* out_enc_boxes_ = nullptr;   // [B, nq, 4]
  int* topk_idx_ = nullptr;          // [B, nq]
};

// host helpers exposed for CPU tests
void bicubic_resize_chlast(const float* src, int n_in, int C, int n_out, float* dst);   // [n_in,n_in,C] -> [n_out,n_out,C]

}  // namespace lwb
