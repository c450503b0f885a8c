/*
 * lwdetr_b200 - C ABI of the B200-native LW-DETR inference path.
 *
 * Every entry point takes plain pointers and sizes (no torch types).  Device pointers are CUDA
 * device addresses on the current device; `stream` is a cudaStream_t passed as void* (NULL = the
 * legacy default stream).  All calls are stream-ordered and asynchronous unless stated otherwise.
 * Return value: 0 on success, non-zero on failure with a message in lwdetr_last_error()
 * (thread-local).  Nothing throws across this boundary.
 *
 * The reference interface each group replaces is cited as file:line relative to the
 * Atten4Vis/LW-DETR tree.
 */
#ifndef LWDETR_B200_H_
#define LWDETR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LWDETR_API __attribute__((visibility("default")))

enum { LWDETR_F16 = 0, LWDETR_BF16 = 1 };
enum { LWDETR_ACT_NONE = 0, LWDETR_ACT_RELU = 1, LWDETR_ACT_GELU = 2, LWDETR_ACT_SILU = 3 };

LWDETR_API const char* lwdetr_last_error(void);
/* Debug aid: with LWDETR_B200_DEBUG_WAIT=1 in the environment the attention kernel's barrier waits time out after ~50 ms and
 * record where; this prints the records to stderr (they live in mapped host memory and survive the device fault). */
LWDETR_API int lwdetr_debug_dump(void);
LWDETR_API int lwdetr_abi_version(void);

/* ------------------------------------------------------------------------------------------------
 * Kernel-level entry points (unit tests, ncu captures).  They are the same kernels the model-level
 * forward schedules.
 * ---------------------------------------------------------------------------------------------- */

/* out[rowmap(m), n] = resid[m', n] + gamma[n] * act(sum_k A[m,k] W[n,k] + bias[n])
 * tcgen05/TMA GEMM standing in for F.linear / 1x1 conv / ConvTranspose2d(k2,s2)
 * (models/backbone/vit.py:120-140,206-220; projector.py:85-98,165-190; transformer.py:27-39).
 *   A [M, lda] 16-bit, W [N, K] 16-bit, K % 64 == 0, bias/gamma fp32 [N] or NULL,
 *   resid 16-bit [*, ld_resid] or NULL (row m % resid_mod when resid_mod > 0),
 *   out 16-bit (out_fp32 = 0) or fp32 [*, ld_out].
 *   rows_in = 1: rows are window-major tokens (b, win 4x4, t) of an IH x IW grid (vit.py:353-358);
 *   remap_rows = 1: write rows in spatial (b, y, x) order (the un-windowing of vit.py:362-364);
 *   shuffle_cout > 0: N == 4*cout, column (dy*2+dx)*cout+co goes to pixel (2y+dy, 2x+dx), channel co. */
LWDETR_API int lwdetr_gemm(int dtype, const void* A, int lda, int M, int K, const void* W, int N,
                           const float* bias, const float* gamma, const void* resid, int ld_resid, int resid_mod,
                           int act, void* out, int ld_out, int out_fp32, int rows_in, int remap_rows,
                           int shuffle_cout, int IH, int IW, void* stream);

/* 3x3 convolution, padding 1, stride 1 or 2, NHWC, as an implicit GEMM (no im2col buffer):
 * X [B, stride*OH, stride*OW, ldx] (channel slice of width Cin), W [N, 9*Cin] with k = (dy*3+dx)*Cin + c,
 * out [B*OH*OW, ld_out].  Stands in for ConvX (projector.py:85-98) with BN folded into W/bias. */
LWDETR_API int lwdetr_conv3x3(int dtype, const void* X, int ldx, int B, int OH, int OW, int stride, int Cin,
                              const void* W, int N, const float* bias, int act, void* out, int ld_out,
                              void* stream);

/* LayerNorm over the last dimension of rows (vit.py:198,217 eps 1e-6; projector.py:21-47 on NHWC rows;
 * transformer.py norms eps 1e-5).  x/y 16-bit with leading dimensions, w/b fp32 [C], C % 8 == 0, C <= 1024. */
LWDETR_API int lwdetr_layernorm(int dtype, const void* x, int ldx, void* y, int ldy, const float* w, const float* b,
                                float eps, int64_t rows, int C, void* stream);

/* softmax(Q K^T * scale) V for `nseq` independent sequences of `seqlen` tokens and `heads` heads of
 * width dh in {16, 32, 64}; token (s, t) is matrix row s*seqlen + t, head h occupies columns
 * [h*dh, (h+1)*dh).  Window attention: nseq = 16*B, seqlen = 100; global: nseq = B, seqlen = 1600
 * (vit.py:120-140, 195-222); decoder self-attention: nseq = B, seqlen = nq (attention.py:563-606). */
LWDETR_API int lwdetr_attention(int dtype, const void* q, int ldq, const void* k, int ldk, const void* v, int ldv,
                                void* out, int ldo, int nseq, int seqlen, int heads, int dh, float scale,
                                void* stream);

/* Multi-scale deformable attention forward with the REFERENCE OPERATOR'S OWN INTERFACE:
 *   MultiScaleDeformableAttention.ms_deform_attn_forward(value, spatial_shapes, level_start_index, sampling_loc,
 *   attn_weight, im2col_step) -> [B, Lq, M*D]
 *   (models/ops/src/ms_deform_attn.h:19-35, vision.cpp:13-16, cuda/ms_deform_attn_cuda.cu:20-80,
 *   cuda/ms_deform_im2col_cuda.cuh:33-84,237-299; Python caller functions/ms_deform_attn_func.py:28-38).
 * All pointers DEVICE, contiguous, as the reference asserts (ms_deform_attn_cuda.cu:28-38):
 *   value [B, S, M, D], sampling_loc [B, Lq, M, L, P, 2] (x, y normalised), attn_weight [B, Lq, M, L, P] and
 *   out [B, Lq, M*D] share one element type `etype` (LWDETR_ET_F32 / _F16 / _BF16 - the reference compiles float and
 *   double only, ms_deform_attn_cuda.cu:64); spatial_shapes int64 [L, 2] (H, W) and level_start_index int64 [L] are
 *   DEVICE tensors exactly as the reference receives them.  Any D; D % 4 == 0 (fp32) / D % 8 == 0 (16-bit) with
 *   16-byte aligned value / out takes the vectorised kernel, everything else a one-thread-per-channel kernel.
 * Differences from the reference: the caller owns `out` (the reference allocates at::zeros, :54); every element of out
 * is written, so it need not be zeroed; there is no im2col_step batching loop, but the reference's precondition
 * B % min(B, im2col_step) == 0 (:50-52) is still checked so that the error behaviour matches. */
enum { LWDETR_ET_F32 = 0, LWDETR_ET_F16 = 1, LWDETR_ET_BF16 = 2 };
LWDETR_API int lwdetr_ms_deform_attn_forward(int etype, const void* value, const int64_t* spatial_shapes,
                                             const int64_t* level_start_index, const void* sampling_loc,
                                             const void* attn_weight, void* out, int B, int S, int M, int D, int Lq,
                                             int L, int P, int im2col_step, void* stream);

/* Backward of the same operator, fp32 (ms_deform_attn.h:37-60, ms_deform_attn_cuda.cu:83-154, cuh:301-920):
 *   MSDA.ms_deform_attn_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output,
 *   im2col_step) -> [grad_value, grad_sampling_loc, grad_attn_weight].
 * grad_output [B, Lq, M*D]; grad_value [B, S, M, D] is zeroed by the call (the reference returns at::zeros_like, :120) and
 * accumulated with atomicAdd as in the reference; grad_sampling_loc [B, Lq, M, L, P, 2] and grad_attn_weight
 * [B, Lq, M, L, P] are written once per element.  Caller-owned, stream-ordered. */
LWDETR_API int lwdetr_ms_deform_attn_backward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                              const float* sampling_loc, const float* attn_weight, const float* grad_output,
                                              float* grad_value, float* grad_sampling_loc, float* grad_attn_weight, int B, int S,
                                              int M, int D, int Lq, int L, int P, int im2col_step, void* stream);

/* The fused form the model schedules (same arithmetic, fewer bytes): the softmax over the L*P attention logits and the
 * sampling-location arithmetic of MSDeformAttn.forward (ops/modules/ms_deform_attn.py:118-131, 4-d reference boxes) run
 * inside the kernel, which therefore takes the RAW projections, and the value tensor is HEAD-MAJOR so that everything one
 * (image, head) can sample is one contiguous slab streamed through shared memory (csrc/msda.cu):
 *   value_hm     16-bit, element (b, m, s, c) at b*v_image_stride + (m*S + s)*16 + c   (D = 16)
 *   offs_logits  16-bit [B*Lq, ld_ol] = [M*L*P*2 sampling offsets | M*L*P attention logits]
 *   ref          fp32   [B*Lq, 4]     reference boxes (cx, cy, w, h)
 *   valid_ratio  fp32   [B, L, 2] (w, h) or NULL: per-level valid ratios of a padded batch
 *                (transformer.py:189-196, 352-353)
 *   spatial_shapes int32 [L, 2] (H, W) and level_start_index int32 [L] on the HOST
 *   out          16-bit [B*Lq, ld_out] */
LWDETR_API int lwdetr_msda_forward(int dtype, const void* value_hm, int64_t v_image_stride, const void* offs_logits,
                                   int ld_ol, const float* ref, const float* valid_ratio, void* out, int ld_out, int B,
                                   int S, int Lq, int M, int L, int P, const int32_t* spatial_shapes_host,
                                   const int32_t* level_start_host, void* stream);

/* torch.topk(score, k, dim=1)[1] for fp32 score [B, S] -> int32 idx [B, k], sorted, ties -> lower index
 * (transformer.py:246). */
LWDETR_API int lwdetr_topk(const float* score, int B, int S, int k, int32_t* idx, void* stream);

/* PostProcess.forward (lwdetr.py:515-544) fused on the device: per image the top `num_select` of
 * sigmoid(pred_logits) over the nq*num_classes (query, class) pairs, sorted descending (ties -> lower flat index, as
 * torch.topk), labels = flat % num_classes, boxes = pred_boxes[flat / num_classes] converted cxcywh -> xyxy and scaled
 * by target_sizes [B,2] = (height, width).  All pointers DEVICE: pred_logits fp32 [B,nq,num_classes], pred_boxes fp32
 * [B,nq,4], target_sizes fp32 [B,2], work int32 [B * ceil(nq*num_classes/16384) * num_select] scratch,
 * scores fp32 [B,num_select], labels int32 [B,num_select], boxes fp32 [B,num_select,4]. */
LWDETR_API int lwdetr_postprocess(const float* pred_logits, const float* pred_boxes, const float* target_sizes, int B, int nq,
                                  int num_classes, int num_select, int32_t* work, float* scores, int32_t* labels, float* boxes,
                                  void* stream);

/* Host helper (no GPU): bicubic, align_corners=False resize of a channels-last [n_in, n_in, C] fp32 grid
 * to [n_out, n_out, C] - the absolute position embedding resize of vit.py:26-54, done once at load. */
LWDETR_API int lwdetr_host_bicubic(const float* src, int n_in, int C, int n_out, float* dst);

/* ------------------------------------------------------------------------------------------------
 * Model-level API: what models.lwdetr.LWDETR.forward (lwdetr.py:111-174) binds to.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lwdetr_handle lwdetr_handle;

typedef struct {
  int32_t vit_dim, vit_depth, vit_heads;
  int32_t window_block_mask;     /* bit i set: block i uses window attention (vit.py:195-222) */
  int32_t n_taps, taps[4];       /* out_feature_indexes, ascending (vit.py:311-316) */
  int32_t n_levels, level_scale_log2[2]; /* projector levels: +1 = P3 (x2), 0 = P4, -1 = P5 (/2) */
  int32_t hidden_dim, sa_heads, ca_heads, dec_points, num_queries, dec_layers, dim_feedforward;
  int32_t num_classes, group_detr, img_size;
} lwdetr_config;

typedef struct {
  float* aux_logits;   /* [dec_layers-1, B, nq, num_classes] or NULL */
  float* aux_boxes;    /* [dec_layers-1, B, nq, 4] or NULL */
  float* enc_logits;   /* [B, nq, num_classes] or NULL */
  float* enc_boxes;    /* [B, nq, 4] or NULL */
  int32_t* topk_index; /* [B, nq] two-stage selection (token index per query slot) or NULL */
} lwdetr_aux_out;

/* One handle per (device, config, compute dtype); not thread-safe per handle.  The handle binds to the CUDA device
 * that is current at creation; every later call switches to that device for its duration. */
LWDETR_API int lwdetr_create(const lwdetr_config* cfg, int dtype, lwdetr_handle** out);
LWDETR_API void lwdetr_destroy(lwdetr_handle* h);

/* Pack the checkpoint: `n` named fp32 HOST tensors with the reference's state_dict names
 * (SURVEY.md 8b).  Folds BatchNorm into the convolutions, merges q/v biases, concatenates the
 * deformable-attention projections, resizes the position embedding to cfg.img_size (the raw table is kept for
 * lwdetr_forward_at), converts to the compute dtype and uploads.  Synchronous.  May be called again after the weights
 * change. */
LWDETR_API int lwdetr_load_weights(lwdetr_handle* h, int n, const char* const* names, const float* const* data,
                                   const int64_t* numel);

/* images: DEVICE [B, 3, S, S] with S = cfg.img_size, fp32 (images_fp32 = 1) or the compute dtype; outputs: DEVICE fp32
 * pred_logits [B, nq, num_classes], pred_boxes [B, nq, 4]; aux may be NULL.  topk_override: DEVICE
 * int32 [B, nq] or NULL - test hook that forces the two-stage selection (SURVEY.md 8c tier T2). */
LWDETR_API int lwdetr_forward(lwdetr_handle* h, const void* images, int images_fp32, int B, float* pred_logits,
                              float* pred_boxes, const lwdetr_aux_out* aux, const int32_t* topk_override,
                              void* stream);

/* The same forward with the two input forms the callers on either side of the path use (SURVEY.md 8f):
 *   format LWDETR_IN_U8_NHWC: images is DEVICE uint8 [B, S, S, 3] - the output of an image decoder + resize.  ToTensor's /255
 *     and Normalize(mean, std) (demo/demo.py:146-159, datasets/transforms.py:223-252) are fused into the patch gather:
 *     (x/255 - mean[c]) / std[c]; the fp32 NCHW image never exists (4x fewer input bytes over PCIe and HBM).
 *   padding_mask: DEVICE bool [B, S, S] (True = padded pixel), the NestedTensor mask of a padded / mixed-size batch
 *     (util/misc.py:317-339), or NULL.  Implements backbone.py:153-158 (nearest resize per level), transformer.py:
 *     86-89,112-123 (per-image proposals, masked memory rows), :189-196,352-355 (valid ratios on the reference boxes) and
 *     ops/modules/ms_deform_attn.py:114-115 (masked value rows).  The ViT itself takes no mask (backbone.py:145). */
enum { LWDETR_IN_F32_NCHW = 0, LWDETR_IN_16_NCHW = 1, LWDETR_IN_U8_NHWC = 2 };
typedef struct {
  const void* images;
  int32_t format;
  const uint8_t* padding_mask;
  float mean[3], std[3];        /* LWDETR_IN_U8_NHWC only */
} lwdetr_input;
LWDETR_API int lwdetr_forward_ex(lwdetr_handle* h, const lwdetr_input* input, int B, float* pred_logits, float* pred_boxes,
                                 const lwdetr_aux_out* aux, const int32_t* topk_override, void* stream);

/* The same forward on uint8 RGB frames of ANY size, each resized on the device exactly as the reference's callers resize
 * on the host: demo/demo.py:146-159 runs transforms.Resize([640, 640]) on a PIL image, and the square_resize_div_64 eval
 * transform (datasets/transforms.py:223-232, datasets/coco.py:149-153) is the same call.  Both are Pillow's
 * Image.resize((S, S), BILINEAR); the result here is bit-identical to it (csrc/resize.cu states the arithmetic), and
 * the /255, Normalize(mean, std) and patch gather of LWDETR_IN_U8_NHWC follow in the same kernel.  So the predictions
 * are bit-identical to lwdetr_forward_at on the Pillow-resized frames, and the resize costs no host time.
 *   frames: HOST array [B] of descriptors; each frame's pixels are DEVICE HWC RGB uint8, pixel (y, x) channel c at
 *     data + y*row_stride + x*3 + c.  Sides in [1, LWDETR_MAX_FRAME_SIDE], row_stride >= 3*width (cropped views need
 *     no copy), no alignment requirement; one batch may mix sizes.  B <= LWDETR_MAX_FRAMES (descriptors travel as kernel
 *     parameters).  The frames must stay valid until the stream has consumed them.
 *   img_size follows the rule of lwdetr_forward_at.  frames and lwdetr_forward_at share one schedule (and CUDA graph)
 *   per (B, img_size): frames of new sizes need no re-plan.  Boxes come out normalised to the frame, as the
 *   reference's do; scale them by each frame's (height, width) (PostProcess target_sizes) for source pixels. */
#define LWDETR_MAX_FRAMES 1024
#define LWDETR_MAX_FRAME_SIDE 8192
typedef struct {
  const uint8_t* data;   /* DEVICE, HWC RGB */
  int32_t height, width;
  int64_t row_stride;    /* bytes */
} lwdetr_frame;
LWDETR_API int lwdetr_forward_frames(lwdetr_handle* h, const lwdetr_frame* frames, int B, int img_size, const float mean[3],
                                     const float std[3], float* pred_logits, float* pred_boxes, const lwdetr_aux_out* aux,
                                     const int32_t* topk_override, void* stream);

/* The same forward at a chosen square input resolution: images (and padding_mask) are [B, ., img_size, img_size] with
 * img_size a multiple of 64 in [LWDETR_MIN_IMG_SIZE, LWDETR_MAX_IMG_SIZE] - the sizes the reference trains its models
 * at (datasets/coco.py:133, square_resize_div_64) - or the handle's cfg.img_size.  The ViT runs on an (img_size/16)^2
 * token grid with the position embedding resized to it (vit.py:26-54, 343-365); projector levels, proposals and the
 * deformable attention follow the feature map sizes.  One handle serves every resolution from one weight arena: a
 * change of (B, img_size) re-plans the schedule (and drops its CUDA graphs), exactly as a change of B does.
 * lwdetr_forward_ex(h, ...) is lwdetr_forward_at(h, ..., cfg.img_size, ...). */
#define LWDETR_MIN_IMG_SIZE 448
#define LWDETR_MAX_IMG_SIZE 896
LWDETR_API int lwdetr_forward_at(lwdetr_handle* h, const lwdetr_input* input, int img_size, int B, float* pred_logits,
                                 float* pred_boxes, const lwdetr_aux_out* aux, const int32_t* topk_override, void* stream);

/* Multi-GPU init (SURVEY.md 8e): ONE ncclBroadcast of the packed weight arena from rank `root`, stream-ordered on
 * `stream`; the only collective of the path (images shard across ranks as independent replicas, nothing on the hot path).
 * Every rank first calls lwdetr_load_weights with tensors of the right shapes (any values on the non-root ranks): that
 * fixes the arena layout, which is a function of (config, dtype) only; the call verifies that the arena sizes agree.
 * On success the handle's schedule is re-planned at its next forward (position tables follow the received weights).
 * `nccl_comm` is an ncclComm_t of a communicator the caller created (one rank per GPU); NCCL is resolved at run time
 * from the libnccl already loaded in the process (or dlopen("libnccl.so.2")), the library does not link it. */
LWDETR_API int lwdetr_broadcast_weights(lwdetr_handle* h, void* nccl_comm, int root, void* stream);
LWDETR_API int64_t lwdetr_weight_arena_bytes(lwdetr_handle* h);

/* options: "cuda_graph" (0/1, default 0: the caller opts in after warm-up), "fuse_layernorm" (0/1, default 1), "pdl" (0/1, default 1: programmatic dependent
 * launch of every kernel; process-wide) */
LWDETR_API int lwdetr_set_option(lwdetr_handle* h, const char* name, int value);

/* Debug captures (tests): after the op labelled `label` runs in the next forward, its output is copied to
 * the HOST buffer dst as fp32 (row-major, dense).  lwdetr_capture_result returns the element count. */
LWDETR_API int lwdetr_add_capture(lwdetr_handle* h, const char* label, float* dst, int64_t capacity);
LWDETR_API int64_t lwdetr_capture_result(lwdetr_handle* h, int index);
LWDETR_API void lwdetr_clear_captures(lwdetr_handle* h);

/* Schedule introspection / per-op timing of the last planned batch size.  The bytes of the input-reading op
 * "patch_gather" are those of the last forward's input (after lwdetr_forward_frames: the frames' bytes). */
LWDETR_API int lwdetr_num_ops(lwdetr_handle* h);
LWDETR_API const char* lwdetr_op_label(lwdetr_handle* h, int i);
LWDETR_API int lwdetr_op_cost(lwdetr_handle* h, int i, double* flops, double* bytes);
LWDETR_API int lwdetr_profile_ops(lwdetr_handle* h, int iters, float* ms_per_op, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LWDETR_B200_H_ */
