// C-ABI surface (include/lwdetr_b200.h): argument checking, error strings, dispatch to the kernels.
#include "lwdetr_b200.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdint.h>

#include <string>

#include <map>
#include <new>
#include <vector>

#include "attn.h"
#include "engine.h"
#include "gemm_tc.h"
#include "msda.h"
#include "rowops.h"

namespace lwb { int attention_slots_debug_dump(); }   // attn_slots.cu

namespace {
thread_local std::string g_err;
int fail(const std::string& m) {
  g_err = m;
  return -1;
}
int cuda_fail(int e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(static_cast<cudaError_t>(e));
  return -1;
}
}  // namespace

extern "C" {

const char* lwdetr_last_error(void) { return g_err.c_str(); }
int lwdetr_abi_version(void) { return 1; }

int lwdetr_gemm(int dtype, const void* A, int lda, int M, int K, const void* W, int N, const float* bias,
                const float* gamma, const void* resid, int ld_resid, int resid_mod, int act, void* out, int ld_out,
                int out_fp32, int rows_in, int remap_rows, int shuffle_cout, int IH, int IW, void* stream) {
  if (!A || !W || !out) return fail("lwdetr_gemm: null pointer");
  lwb::GemmDesc d;
  d.dtype = dtype; d.A = A; d.lda = lda; d.M = M; d.N = N; d.K = K; d.W = W; d.bias = bias; d.gamma = gamma;
  d.resid = resid; d.ld_resid = ld_resid; d.resid_mod = resid_mod; d.act = act; d.out = out; d.ld_out = ld_out;
  d.out_fp32 = out_fp32; d.rows_in = rows_in; d.remap_rows = remap_rows; d.shuffle_cout = shuffle_cout;
  d.IH = IH; d.IW = IW;
  lwb::GemmOp op;
  std::string err;
  if (lwb::gemm_build(d, &op, &err)) return fail("lwdetr_gemm: " + err);
  int e = lwb::gemm_launch(op, static_cast<cudaStream_t>(stream));
  if (e) return cuda_fail(e, "lwdetr_gemm launch");
  return 0;
}

int lwdetr_conv3x3(int dtype, const void* X, int ldx, int B, int OH, int OW, int stride, int Cin, const void* W,
                   int N, const float* bias, int act, void* out, int ld_out, void* stream) {
  if (!X || !W || !out) return fail("lwdetr_conv3x3: null pointer");
  if (stride != 1 && stride != 2) return fail("lwdetr_conv3x3: stride must be 1 or 2");
  lwb::GemmDesc d;
  d.dtype = dtype; d.a_mode = stride == 1 ? lwb::AMODE_CONV3_S1 : lwb::AMODE_CONV3_S2;
  d.A = X; d.lda = ldx; d.B = B; d.OH = OH; d.OW = OW; d.M = B * OH * OW; d.N = N; d.K = 9 * Cin; d.W = W;
  d.bias = bias; d.act = act; d.out = out; d.ld_out = ld_out;
  lwb::GemmOp op;
  std::string err;
  if (lwb::gemm_build(d, &op, &err)) return fail("lwdetr_conv3x3: " + err);
  int e = lwb::gemm_launch(op, static_cast<cudaStream_t>(stream));
  if (e) return cuda_fail(e, "lwdetr_conv3x3 launch");
  return 0;
}


int lwdetr_layernorm(int dtype, const void* x, int ldx, void* y, int ldy, const float* w, const float* b, float eps,
                     int64_t rows, int C, void* stream) {
  if (!x || !y || !w || !b) return fail("lwdetr_layernorm: null pointer");
  lwb::LayerNormArgs a{};
  a.x = x; a.ldx = ldx; a.y = y; a.ldy = ldy; a.w = w; a.b = b; a.eps = eps; a.rows = rows; a.C = C; a.flag_mod = 1;
  int e = lwb::layernorm_launch(dtype, a, static_cast<cudaStream_t>(stream));
  if (e == -2) return fail("lwdetr_layernorm: C must be a multiple of 8 and <= 1024");
  if (e) return cuda_fail(e, "lwdetr_layernorm launch");
  return 0;
}

int lwdetr_attention(int dtype, const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* out, int ldo,
                     int nseq, int seqlen, int heads, int dh, float scale, void* stream) {
  if (!q || !k || !v || !out) return fail("lwdetr_attention: null pointer");
  if ((ldq | ldk | ldv | ldo) % 8) return fail("lwdetr_attention: leading dimensions must be multiples of 8");
  lwb::AttnArgs a{};
  a.q = q; a.k = k; a.v = v; a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.o = out; a.ldo = ldo; a.seqlen = seqlen; a.nseq = nseq;
  a.heads = heads; a.scale_log2 = scale * 1.4426950408889634f;
  int e = lwb::attention_launch(dtype, a, dh, static_cast<cudaStream_t>(stream));
  if (e == -2) return fail("lwdetr_attention: head dim must be 16, 32 or 64");
  if (e) return cuda_fail(e, "lwdetr_attention launch");
  return 0;
}

int lwdetr_ms_deform_attn_forward(int etype, const void* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                  const void* sampling_loc, const void* attn_weight, void* out, int B, int S, int M, int D, int Lq, int L,
                                  int P, int im2col_step, void* stream) {
  if (!value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight || !out) return fail("lwdetr_ms_deform_attn_forward: null pointer");
  if (etype != LWDETR_ET_F32 && etype != LWDETR_ET_F16 && etype != LWDETR_ET_BF16) return fail("lwdetr_ms_deform_attn_forward: etype must be LWDETR_ET_F32, _F16 or _BF16");
  if (B < 1 || S < 1 || M < 1 || D < 1 || Lq < 1 || L < 1 || P < 1) return fail("lwdetr_ms_deform_attn_forward: sizes must be positive");
  if (im2col_step < 1 || B % (B < im2col_step ? B : im2col_step) != 0)
    return fail("lwdetr_ms_deform_attn_forward: batch(" + std::to_string(B) + ") must divide im2col_step(" + std::to_string(im2col_step) + ")");   // ms_deform_attn_cuda.cu:50-52
  lwb::MsdaOpArgs a{};
  a.value = value; a.spatial_shapes = spatial_shapes; a.level_start_index = level_start_index; a.sampling_loc = sampling_loc;
  a.attn_weight = attn_weight; a.out = out; a.B = B; a.S = S; a.M = M; a.D = D; a.Lq = Lq; a.L = L; a.P = P;
  int e = lwb::msda_op_launch(etype, a, static_cast<cudaStream_t>(stream));
  if (e == -2) return fail("lwdetr_ms_deform_attn_forward: unsupported element type / head dim");
  if (e) return cuda_fail(e, "lwdetr_ms_deform_attn_forward launch");
  return 0;
}

int lwdetr_ms_deform_attn_backward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index, const float* sampling_loc,
                                   const float* attn_weight, const float* grad_output, float* grad_value, float* grad_sampling_loc,
                                   float* grad_attn_weight, int B, int S, int M, int D, int Lq, int L, int P, int im2col_step, void* stream) {
  if (!value || !spatial_shapes || !level_start_index || !sampling_loc || !attn_weight || !grad_output || !grad_value || !grad_sampling_loc || !grad_attn_weight)
    return fail("lwdetr_ms_deform_attn_backward: null pointer");
  if (B < 1 || S < 1 || M < 1 || D < 1 || Lq < 1 || L < 1 || P < 1) return fail("lwdetr_ms_deform_attn_backward: sizes must be positive");
  if (im2col_step < 1 || B % (B < im2col_step ? B : im2col_step) != 0)
    return fail("lwdetr_ms_deform_attn_backward: batch(" + std::to_string(B) + ") must divide im2col_step(" + std::to_string(im2col_step) + ")");   // ms_deform_attn_cuda.cu:116-118
  lwb::MsdaOpArgs a{};
  a.value = value; a.spatial_shapes = spatial_shapes; a.level_start_index = level_start_index; a.sampling_loc = sampling_loc;
  a.attn_weight = attn_weight; a.out = nullptr; a.B = B; a.S = S; a.M = M; a.D = D; a.Lq = Lq; a.L = L; a.P = P;
  int e = lwb::msda_op_backward_launch(a, grad_output, grad_value, grad_sampling_loc, grad_attn_weight, static_cast<cudaStream_t>(stream));
  if (e) return cuda_fail(e, "lwdetr_ms_deform_attn_backward launch");
  return 0;
}

int lwdetr_debug_dump(void) { return lwb::attention_slots_debug_dump(); }

int lwdetr_msda_forward(int dtype, const void* value_hm, int64_t v_image_stride, const void* offs_logits, int ld_ol, const float* ref,
                        const float* valid_ratio, void* out, int ld_out, int B, int S, int Lq, int M, int L, int P,
                        const int32_t* spatial_shapes_host, const int32_t* level_start_host, void* stream) {
  if (!value_hm || !offs_logits || !ref || !out || !spatial_shapes_host || !level_start_host) return fail("lwdetr_msda_forward: null pointer");
  if (L < 1 || L > lwb::MSDA_MAX_LEVELS) return fail("lwdetr_msda_forward: 1..4 levels supported");
  if ((ld_out % 8) || (ld_ol % 2) || (v_image_stride % 8) || (reinterpret_cast<uintptr_t>(value_hm) & 15)) return fail("lwdetr_msda_forward: misaligned leading dimension / base");
  if (v_image_stride < static_cast<int64_t>(M) * S * lwb::MSDA_D) return fail("lwdetr_msda_forward: v_image_stride smaller than one image's M*S*16 values");
  lwb::MsdaArgs a{};
  a.value = value_hm; a.v_b_stride = v_image_stride; a.offs_logits = offs_logits; a.ld_ol = ld_ol; a.ref = ref; a.valid_ratio = valid_ratio;
  a.out = out; a.ld_out = ld_out; a.batch = B; a.nq = Lq; a.heads = M; a.levels = L; a.points = P; a.S = S;
  for (int l = 0; l < L; ++l) { a.lvl_h[l] = spatial_shapes_host[2 * l]; a.lvl_w[l] = spatial_shapes_host[2 * l + 1]; a.lvl_start[l] = level_start_host[l]; }
  if (lwb::msda_plan(&a)) return fail("lwdetr_msda_forward: a feature level is wider than 840 tokens, larger than 16384 tokens, or there are too many bands");
  int e = lwb::msda_launch(dtype, a, static_cast<cudaStream_t>(stream));
  if (e == -2) return fail("lwdetr_msda_forward: unsupported (levels, points) combination");
  if (e) return cuda_fail(e, "lwdetr_msda_forward launch");
  return 0;
}

int lwdetr_topk(const float* score, int B, int S, int k, int32_t* idx, void* stream) {
  if (!score || !idx) return fail("lwdetr_topk: null pointer");
  int e = lwb::topk_launch(score, B, S, k, idx, static_cast<cudaStream_t>(stream));
  if (e == -2) return fail("lwdetr_topk: need k <= S <= 16384");
  if (e) return cuda_fail(e, "lwdetr_topk launch");
  return 0;
}

int lwdetr_postprocess(const float* pred_logits, const float* pred_boxes, const float* target_sizes, int B, int nq, int num_classes,
                       int num_select, int32_t* work, float* scores, int32_t* labels, float* boxes, void* stream) {
  if (!pred_logits || !pred_boxes || !target_sizes || !work || !scores || !labels || !boxes) return fail("lwdetr_postprocess: null pointer");
  if (B < 1 || nq < 1 || num_classes < 1 || num_select < 1) return fail("lwdetr_postprocess: bad sizes");
  int e = lwb::postprocess_launch(pred_logits, pred_boxes, target_sizes, B, nq, num_classes, num_select, work, scores, labels, boxes,
                                  static_cast<cudaStream_t>(stream));
  if (e == -2) return fail("lwdetr_postprocess: need num_select <= slice length and slices * num_select <= 16384");
  if (e) return cuda_fail(e, "lwdetr_postprocess launch");
  return 0;
}

int lwdetr_host_bicubic(const float* src, int n_in, int C, int n_out, float* dst) {
  if (!src || !dst || n_in < 1 || n_out < 1 || C < 1) return fail("lwdetr_host_bicubic: bad arguments");
  lwb::bicubic_resize_chlast(src, n_in, C, n_out, dst);
  return 0;
}

// ------------------------------------------------------------------------------------------ model level
struct lwdetr_handle {
  lwb::Engine* eng;
};

int lwdetr_create(const lwdetr_config* cfg, int dtype, lwdetr_handle** out) {
  if (!cfg || !out) return fail("lwdetr_create: null pointer");
  if (dtype != LWDETR_F16 && dtype != LWDETR_BF16) return fail("lwdetr_create: dtype must be LWDETR_F16 or LWDETR_BF16");
  if (cfg->n_taps < 1 || cfg->n_taps > 4 || cfg->n_levels < 1 || cfg->n_levels > 2 || cfg->vit_depth < 1 || cfg->vit_depth > 31)
    return fail("lwdetr_create: unsupported configuration");
  if (cfg->img_size % 64 != 0 || cfg->vit_dim % 64 != 0 || cfg->hidden_dim % 128 != 0)
    return fail("lwdetr_create: img_size % 64, vit_dim % 64 and hidden_dim % 128 must be 0");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("lwdetr_create: no CUDA device (there is no CPU fallback)");
  if (cfg->num_classes < 1 || cfg->num_classes > 4096) return fail("lwdetr_create: num_classes must be in [1, 4096]");
  lwdetr_handle* h = new (std::nothrow) lwdetr_handle;
  if (!h) return fail("lwdetr_create: out of memory");
  h->eng = new (std::nothrow) lwb::Engine(*cfg, dtype);
  if (!h->eng) { delete h; return fail("lwdetr_create: out of memory"); }
  *out = h;
  return 0;
}

void lwdetr_destroy(lwdetr_handle* h) {
  if (!h) return;
  delete h->eng;
  delete h;
}

int lwdetr_load_weights(lwdetr_handle* h, int n, const char* const* names, const float* const* data, const int64_t* numel) {
  if (!h || !names || !data || !numel) return fail("lwdetr_load_weights: null pointer");
  std::map<std::string, lwb::HostTensor> m;
  for (int i = 0; i < n; ++i) m[names[i]] = lwb::HostTensor{data[i], numel[i]};
  std::string err;
  if (h->eng->load_weights(m, &err)) return fail("lwdetr_load_weights: " + err);
  return 0;
}

int lwdetr_forward(lwdetr_handle* h, const void* images, int images_fp32, int B, float* pred_logits, float* pred_boxes,
                   const lwdetr_aux_out* aux, const int32_t* topk_override, void* stream) {
  if (!h || !images) return fail("lwdetr_forward: null pointer");
  std::string err;
  lwb::ForwardIn in;
  in.images = images; in.kind = images_fp32 ? lwb::IN_F32_NCHW : lwb::IN_16_NCHW;
  if (h->eng->forward(in, B, h->eng->config().img_size, pred_logits, pred_boxes, aux, topk_override, static_cast<cudaStream_t>(stream), &err))
    return fail(err);
  return 0;
}

int lwdetr_forward_at(lwdetr_handle* h, const lwdetr_input* input, int img_size, int B, float* pred_logits, float* pred_boxes,
                      const lwdetr_aux_out* aux, const int32_t* topk_override, void* stream) {
  if (!h || !input || !input->images) return fail("lwdetr_forward_at: null pointer");
  if (input->format != LWDETR_IN_F32_NCHW && input->format != LWDETR_IN_16_NCHW && input->format != LWDETR_IN_U8_NHWC)
    return fail("lwdetr_forward_at: format must be LWDETR_IN_F32_NCHW, LWDETR_IN_16_NCHW or LWDETR_IN_U8_NHWC");
  const bool in_range = img_size >= LWDETR_MIN_IMG_SIZE && img_size <= LWDETR_MAX_IMG_SIZE && img_size % 64 == 0;
  if (!in_range && img_size != h->eng->config().img_size)
    return fail("lwdetr_forward_at: img_size " + std::to_string(img_size) + " is neither a multiple of 64 in [" +
                std::to_string(LWDETR_MIN_IMG_SIZE) + ", " + std::to_string(LWDETR_MAX_IMG_SIZE) + "] nor the handle's img_size " +
                std::to_string(h->eng->config().img_size));
  lwb::ForwardIn in;
  in.images = input->images; in.kind = input->format; in.mask = input->padding_mask;
  for (int c = 0; c < 3; ++c) {
    in.mean[c] = input->mean[c]; in.stdv[c] = input->std[c];
    if (input->format == LWDETR_IN_U8_NHWC && !(input->std[c] > 0.f)) return fail("lwdetr_forward_at: std must be positive");
  }
  std::string err;
  if (h->eng->forward(in, B, img_size, pred_logits, pred_boxes, aux, topk_override, static_cast<cudaStream_t>(stream), &err)) return fail(err);
  return 0;
}

int lwdetr_forward_frames(lwdetr_handle* h, const lwdetr_frame* frames, int B, int img_size, const float mean[3], const float std[3],
                          float* pred_logits, float* pred_boxes, const lwdetr_aux_out* aux, const int32_t* topk_override, void* stream) {
  if (!h || !frames || !mean || !std) return fail("lwdetr_forward_frames: null pointer");
  if (B < 1 || B > LWDETR_MAX_FRAMES)
    return fail("lwdetr_forward_frames: B = " + std::to_string(B) + " is outside [1, " + std::to_string(LWDETR_MAX_FRAMES) + "]");
  const bool in_range = img_size >= LWDETR_MIN_IMG_SIZE && img_size <= LWDETR_MAX_IMG_SIZE && img_size % 64 == 0;
  if (!in_range && img_size != h->eng->config().img_size)
    return fail("lwdetr_forward_frames: img_size " + std::to_string(img_size) + " is neither a multiple of 64 in [" +
                std::to_string(LWDETR_MIN_IMG_SIZE) + ", " + std::to_string(LWDETR_MAX_IMG_SIZE) + "] nor the handle's img_size " +
                std::to_string(h->eng->config().img_size));
  for (int i = 0; i < B; ++i) {
    const lwdetr_frame& f = frames[i];
    const std::string which = "lwdetr_forward_frames: frame " + std::to_string(i);
    if (!f.data) return fail(which + " has a null data pointer");
    if (f.height < 1 || f.width < 1 || f.height > LWDETR_MAX_FRAME_SIDE || f.width > LWDETR_MAX_FRAME_SIDE)
      return fail(which + " is " + std::to_string(f.height) + " x " + std::to_string(f.width) + "; sides must be in [1, " +
                  std::to_string(LWDETR_MAX_FRAME_SIDE) + "]");
    if (f.row_stride < 3LL * f.width)
      return fail(which + ": row_stride " + std::to_string(f.row_stride) + " is less than 3 * width = " + std::to_string(3LL * f.width));
  }
  lwb::ForwardIn in;
  in.kind = lwb::IN_U8_FRAMES; in.frames = frames;
  for (int c = 0; c < 3; ++c) {
    in.mean[c] = mean[c]; in.stdv[c] = std[c];
    if (!(std[c] > 0.f)) return fail("lwdetr_forward_frames: std must be positive");
  }
  std::string err;
  if (h->eng->forward(in, B, img_size, pred_logits, pred_boxes, aux, topk_override, static_cast<cudaStream_t>(stream), &err)) return fail(err);
  return 0;
}

int lwdetr_forward_ex(lwdetr_handle* h, const lwdetr_input* input, int B, float* pred_logits, float* pred_boxes,
                      const lwdetr_aux_out* aux, const int32_t* topk_override, void* stream) {
  if (!h) return fail("lwdetr_forward_ex: null pointer");
  return lwdetr_forward_at(h, input, h->eng->config().img_size, B, pred_logits, pred_boxes, aux, topk_override, stream);
}

// One ncclBroadcast of the packed weight arena (SURVEY.md 8b / 8e).  NCCL is not linked: the symbol is taken from the
// libnccl the host process already loaded (torch's bundled libnccl.so.2) or dlopen'ed by soname.
int lwdetr_broadcast_weights(lwdetr_handle* h, void* nccl_comm, int root, void* stream) {
  if (!h || !nccl_comm) return fail("lwdetr_broadcast_weights: null pointer");
  if (!h->eng->weights_loaded()) return fail("lwdetr_broadcast_weights: call lwdetr_load_weights on every rank first (it fixes the arena layout)");
  typedef int (*PFN_bcast)(const void*, void*, size_t, int, int, void*, cudaStream_t);
  static PFN_bcast fn = nullptr;
  if (!fn) {
    void* sym = dlsym(RTLD_DEFAULT, "ncclBroadcast");
    if (!sym) {
      void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
      if (lib) sym = dlsym(lib, "ncclBroadcast");
    }
    if (!sym) return fail("lwdetr_broadcast_weights: ncclBroadcast not found (load libnccl.so.2 into the process first)");
    fn = reinterpret_cast<PFN_bcast>(sym);
  }
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(h->eng->device());
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // layout check: every rank must hold an arena of the root's size (same config, dtype and library version)
  unsigned long long* dsz = nullptr;
  unsigned long long mine = h->eng->arena_used(), roots = 0;
  int rc = 0;
  if (cudaMalloc(&dsz, 8) != cudaSuccess) rc = -1;
  if (!rc && cudaMemcpyAsync(dsz, &mine, 8, cudaMemcpyHostToDevice, st) != cudaSuccess) rc = -1;
  if (!rc && fn(dsz, dsz, 8, /*ncclChar*/ 0, root, nccl_comm, st) != 0) rc = -2;
  if (!rc && cudaMemcpyAsync(&roots, dsz, 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -1;
  if (!rc && cudaStreamSynchronize(st) != cudaSuccess) rc = -1;
  if (dsz) cudaFree(dsz);
  if (!rc && roots != mine) rc = -3;
  if (!rc && fn(h->eng->arena_ptr(), h->eng->arena_ptr(), h->eng->arena_used(), 0, root, nccl_comm, st) != 0) rc = -2;
  cudaSetDevice(prev);
  if (rc == -1) return fail(std::string("lwdetr_broadcast_weights: CUDA error: ") + cudaGetErrorString(cudaGetLastError()));
  if (rc == -2) return fail("lwdetr_broadcast_weights: ncclBroadcast failed");
  if (rc == -3) return fail("lwdetr_broadcast_weights: arena size differs from the root's (" + std::to_string(mine) + " vs " + std::to_string(roots) + " bytes): config / dtype mismatch between ranks");
  h->eng->invalidate_plan();   // a position table planned for another resolution was built from this rank's old weights
  return 0;
}

int64_t lwdetr_weight_arena_bytes(lwdetr_handle* h) { return h ? static_cast<int64_t>(h->eng->arena_used()) : -1; }

int lwdetr_set_option(lwdetr_handle* h, const char* name, int value) {
  if (!h || !name) return fail("lwdetr_set_option: null pointer");
  if (h->eng->set_option(name, value)) return fail(std::string("lwdetr_set_option: unknown option ") + name);
  return 0;
}

int lwdetr_add_capture(lwdetr_handle* h, const char* label, float* dst, int64_t capacity) {
  if (!h || !label || !dst) return fail("lwdetr_add_capture: null pointer");
  h->eng->add_capture(label, dst, capacity);
  return 0;
}
int64_t lwdetr_capture_result(lwdetr_handle* h, int index) { return h ? h->eng->capture_written(index) : -1; }
void lwdetr_clear_captures(lwdetr_handle* h) { if (h) h->eng->clear_captures(); }

int lwdetr_num_ops(lwdetr_handle* h) { return h ? h->eng->num_ops() : 0; }
const char* lwdetr_op_label(lwdetr_handle* h, int i) {
  if (!h || i < 0 || i >= h->eng->num_ops()) return "";
  return h->eng->op(i).label.c_str();
}
int lwdetr_op_cost(lwdetr_handle* h, int i, double* flops, double* bytes) {
  if (!h || i < 0 || i >= h->eng->num_ops()) return fail("lwdetr_op_cost: bad index");
  if (flops) *flops = h->eng->op(i).flops;
  if (bytes) *bytes = h->eng->op(i).bytes;
  return 0;
}
int lwdetr_profile_ops(lwdetr_handle* h, int iters, float* ms_per_op, void* stream) {
  if (!h || !ms_per_op || iters < 1) return fail("lwdetr_profile_ops: bad arguments");
  std::vector<float> ms;
  std::string err;
  if (h->eng->profile_ops(iters, &ms, static_cast<cudaStream_t>(stream), &err)) return fail(err);
  for (size_t i = 0; i < ms.size(); ++i) ms_per_op[i] = ms[i];
  return 0;
}

}  // extern "C"
