"""ctypes binding of include/lwdetr_b200.h.

The shared library is built in-tree by tools/build.py (``__graft_entry__.build()``).  There is no
fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os

from .config import MAX_IMG_SIZE, MIN_IMG_SIZE, input_resolution

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "liblwdetr_b200.so")

F16, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_GELU, ACT_SILU = 0, 1, 2, 3

_lib = None

_vp, _i, _f, _i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_int64

_SIGNATURES = {
    "lwdetr_last_error": (ctypes.c_char_p, []),
    "lwdetr_abi_version": (_i, []),
    "lwdetr_debug_dump": (_i, []),
    "lwdetr_gemm": (_i, [_i, _vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "lwdetr_conv3x3": (_i, [_i, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _vp]),
    "lwdetr_layernorm": (_i, [_i, _vp, _i, _vp, _i, _vp, _vp, _f, _i64, _i, _vp]),
    "lwdetr_attention": (_i, [_i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "lwdetr_ms_deform_attn_forward": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "lwdetr_ms_deform_attn_backward": (_i, [_vp] * 9 + [_i] * 8 + [_vp]),
    "lwdetr_msda_forward": (_i, [_i, _vp, _i64, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "lwdetr_topk": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "lwdetr_postprocess": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "lwdetr_host_bicubic": (_i, [_vp, _i, _i, _i, _vp]),
    "lwdetr_create": (_i, [_vp, _i, _vp]),
    "lwdetr_destroy": (None, [_vp]),
    "lwdetr_load_weights": (_i, [_vp, _i, _vp, _vp, _vp]),
    "lwdetr_forward": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "lwdetr_broadcast_weights": (_i, [_vp, _vp, _i, _vp]),
    "lwdetr_weight_arena_bytes": (_i64, [_vp]),
    "lwdetr_forward_ex": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "lwdetr_forward_at": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "lwdetr_forward_frames": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lwdetr_set_option": (_i, [_vp, ctypes.c_char_p, _i]),
    "lwdetr_add_capture": (_i, [_vp, ctypes.c_char_p, _vp, _i64]),
    "lwdetr_capture_result": (_i64, [_vp, _i]),
    "lwdetr_clear_captures": (None, [_vp]),
    "lwdetr_num_ops": (_i, [_vp]),
    "lwdetr_op_label": (ctypes.c_char_p, [_vp, _i]),
    "lwdetr_op_cost": (_i, [_vp, _i, _vp, _vp]),
    "lwdetr_profile_ops": (_i, [_vp, _i, _vp, _vp]),
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "lwdetr_b200: %s not found - run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / PyTorch fallback)" % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed: %s" % (what, lib().lwdetr_last_error().decode()))


def ptr(t):
    """Device/host address of a torch tensor (or None)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def dtype_code(torch_dtype):
    import torch
    if torch_dtype == torch.float16:
        return F16
    if torch_dtype == torch.bfloat16:
        return BF16
    raise RuntimeError("lwdetr_b200 computes in float16 or bfloat16, got %s" % torch_dtype)


def stream_ptr(device=None):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def gemm(A, W, out, bias=None, gamma=None, resid=None, resid_mod=0, act=ACT_NONE, M=None, K=None, N=None,
         rows_in=0, remap_rows=0, shuffle_cout=0, IH=0, IW=0):
    """out = epilogue(A @ W.T); A [M, K] (row stride A.stride(0)), W [N, K] contiguous."""
    import torch
    M = A.shape[0] if M is None else M
    K = A.shape[1] if K is None else K
    N = W.shape[0] if N is None else N
    check(lib().lwdetr_gemm(dtype_code(A.dtype), ptr(A), A.stride(0), M, K, ptr(W), N, ptr(bias), ptr(gamma),
                            ptr(resid), 0 if resid is None else resid.stride(0), resid_mod, act, ptr(out),
                            out.stride(0), 1 if out.dtype == torch.float32 else 0, rows_in, remap_rows,
                            shuffle_cout, IH, IW, stream_ptr()), "lwdetr_gemm")
    return out


def conv3x3(X, Wk, out, B, OH, OW, stride, Cin, bias=None, act=ACT_NONE):
    """X NHWC [B, s*OH, s*OW, ldx] (uses channels [0, Cin)), Wk [N, 9*Cin], out [B*OH*OW, ld_out]."""
    check(lib().lwdetr_conv3x3(dtype_code(X.dtype), ptr(X), X.stride(2), B, OH, OW, stride, Cin, ptr(Wk),
                               Wk.shape[0], ptr(bias), act, ptr(out), out.stride(0), stream_ptr()),
          "lwdetr_conv3x3")
    return out


def layernorm(x, y, w, b, eps, rows=None, C=None):
    rows = x.shape[0] if rows is None else rows
    C = x.shape[1] if C is None else C
    check(lib().lwdetr_layernorm(dtype_code(x.dtype), ptr(x), x.stride(0), ptr(y), y.stride(0), ptr(w), ptr(b), eps,
                                 rows, C, stream_ptr()), "lwdetr_layernorm")
    return y


def attention(q, k, v, out, nseq, seqlen, heads, dh, scale):
    """q/k/v/out: 2-D views [nseq*seqlen, heads*dh] (any row stride)."""
    check(lib().lwdetr_attention(dtype_code(q.dtype), ptr(q), q.stride(0), ptr(k), k.stride(0), ptr(v), v.stride(0),
                                 ptr(out), out.stride(0), nseq, seqlen, heads, dh, scale, stream_ptr()),
          "lwdetr_attention")
    return out


def value_to_head_major(value, B, S, M):
    """[B*S, M*16] token-major (view, any row stride) -> contiguous head-major [B, M, S, 16] (what value_proj's epilogue writes)."""
    return value.reshape(B, S, M, 16).permute(0, 2, 1, 3).contiguous()


def msda_forward(value_hm, offs_logits, ref, out, B, S, Lq, M, L, P, shapes, valid_ratio=None, v_image_stride=None):
    """value_hm head-major [B, M, S, 16], offs_logits [B*Lq, 3*M*L*P], ref fp32 [B*Lq, 4], out [B*Lq, M*16]."""
    sh = (ctypes.c_int32 * (2 * L))(*[v for hw in shapes for v in hw])
    starts, acc = [], 0
    for h, w in shapes:
        starts.append(acc)
        acc += h * w
    st = (ctypes.c_int32 * L)(*starts)
    stride = M * S * 16 if v_image_stride is None else v_image_stride
    check(lib().lwdetr_msda_forward(dtype_code(value_hm.dtype), ptr(value_hm), stride, ptr(offs_logits),
                                    offs_logits.stride(0), ptr(ref), ptr(valid_ratio), ptr(out), out.stride(0), B, S, Lq, M, L, P,
                                    ctypes.cast(sh, _vp), ctypes.cast(st, _vp), stream_ptr()), "lwdetr_msda_forward")
    return out


ET_F32, ET_F16, ET_BF16 = 0, 1, 2


def ms_deform_attn_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step=64):
    """The reference operator (ms_deform_attn_func.py:28-38 -> MSDA.ms_deform_attn_forward): value [B,S,M,D],
    spatial_shapes int64 [L,2], level_start_index int64 [L], sampling_loc [B,Lq,M,L,P,2], attn_weight [B,Lq,M,L,P], all
    CUDA and contiguous; returns [B, Lq, M*D] in value's dtype (fp32, fp16 or bf16)."""
    import torch
    et = {torch.float32: ET_F32, torch.float16: ET_F16, torch.bfloat16: ET_BF16}.get(value.dtype)
    if et is None:
        raise RuntimeError("ms_deform_attn_forward: value must be float32, float16 or bfloat16, got %s" % value.dtype)
    for name, t in (("value", value), ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index),
                    ("sampling_loc", sampling_loc), ("attn_weight", attn_weight)):
        if not t.is_cuda:
            raise RuntimeError("ms_deform_attn_forward: %s must be a CUDA tensor (Not implemented on the CPU)" % name)   # ms_deform_attn.h:34
        if not t.is_contiguous():
            raise RuntimeError("ms_deform_attn_forward: %s tensor has to be contiguous" % name)                          # ms_deform_attn_cuda.cu:28-32
    if sampling_loc.dtype != value.dtype or attn_weight.dtype != value.dtype:
        raise RuntimeError("ms_deform_attn_forward: value, sampling_loc and attn_weight must share one dtype")
    if spatial_shapes.dtype != torch.int64 or level_start_index.dtype != torch.int64:
        raise RuntimeError("ms_deform_attn_forward: spatial_shapes / level_start_index must be int64")
    B, S, M, D = value.shape
    Lq, L, P = sampling_loc.shape[1], sampling_loc.shape[3], sampling_loc.shape[4]
    out = torch.empty(B, Lq, M * D, device=value.device, dtype=value.dtype)
    check(lib().lwdetr_ms_deform_attn_forward(et, ptr(value), ptr(spatial_shapes), ptr(level_start_index), ptr(sampling_loc),
                                              ptr(attn_weight), ptr(out), B, S, M, D, Lq, L, P, int(im2col_step), stream_ptr()),
          "lwdetr_ms_deform_attn_forward")
    return out


def ms_deform_attn_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output, im2col_step=64):
    """MSDA.ms_deform_attn_backward (ms_deform_attn.h:37-60): fp32 CUDA tensors -> (grad_value, grad_sampling_loc, grad_attn_weight)."""
    import torch
    for name, t in (("value", value), ("sampling_loc", sampling_loc), ("attn_weight", attn_weight), ("grad_output", grad_output)):
        if not t.is_cuda:
            raise RuntimeError("ms_deform_attn_backward: %s must be a CUDA tensor (Not implemented on the CPU)" % name)
        if t.dtype != torch.float32:
            raise RuntimeError("ms_deform_attn_backward: %s must be float32" % name)
        if not t.is_contiguous():
            raise RuntimeError("ms_deform_attn_backward: %s tensor has to be contiguous" % name)
    B, S, M, D = value.shape
    Lq, L, P = sampling_loc.shape[1], sampling_loc.shape[3], sampling_loc.shape[4]
    gv, gl, ga = torch.empty_like(value), torch.empty_like(sampling_loc), torch.empty_like(attn_weight)
    check(lib().lwdetr_ms_deform_attn_backward(ptr(value), ptr(spatial_shapes), ptr(level_start_index), ptr(sampling_loc), ptr(attn_weight),
                                               ptr(grad_output), ptr(gv), ptr(gl), ptr(ga), B, S, M, D, Lq, L, P, int(im2col_step),
                                               stream_ptr()), "lwdetr_ms_deform_attn_backward")
    return gv, gl, ga


def topk(score, k):
    import torch
    B, S = score.shape
    idx = torch.empty(B, k, device=score.device, dtype=torch.int32)
    check(lib().lwdetr_topk(ptr(score), B, S, k, ptr(idx), stream_ptr()), "lwdetr_topk")
    return idx


def postprocess(pred_logits, pred_boxes, target_sizes, num_select):
    """Fused PostProcess (lwdetr.py:515-544) on CUDA fp32 tensors -> (scores [B,k] fp32, labels [B,k] int32, boxes [B,k,4] fp32)."""
    import torch
    B, nq, ncls = pred_logits.shape
    logits = pred_logits.float().contiguous()
    boxes = pred_boxes.float().contiguous()
    ts = target_sizes.to(device=logits.device, dtype=torch.float32).contiguous()
    parts = (nq * ncls + 16383) // 16384
    work = torch.empty(B * parts * num_select, device=logits.device, dtype=torch.int32)
    scores = torch.empty(B, num_select, device=logits.device, dtype=torch.float32)
    labels = torch.empty(B, num_select, device=logits.device, dtype=torch.int32)
    out = torch.empty(B, num_select, 4, device=logits.device, dtype=torch.float32)
    check(lib().lwdetr_postprocess(ptr(logits), ptr(boxes), ptr(ts), B, nq, ncls, num_select, ptr(work), ptr(scores), ptr(labels),
                                   ptr(out), stream_ptr()), "lwdetr_postprocess")
    return scores, labels, out


def host_bicubic(src, n_out):
    """src: CPU fp32 [n, n, C] -> [n_out, n_out, C] (no GPU involved)."""
    import torch
    src = src.contiguous().float()
    dst = torch.empty(n_out, n_out, src.shape[2], dtype=torch.float32)
    check(lib().lwdetr_host_bicubic(ptr(src), src.shape[0], src.shape[2], n_out, ptr(dst)), "lwdetr_host_bicubic")
    return dst


class ConfigStruct(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("vit_dim", "vit_depth", "vit_heads", "window_block_mask", "n_taps")] + \
               [("taps", ctypes.c_int32 * 4), ("n_levels", ctypes.c_int32), ("level_scale_log2", ctypes.c_int32 * 2)] + \
               [(n, ctypes.c_int32) for n in ("hidden_dim", "sa_heads", "ca_heads", "dec_points", "num_queries",
                                              "dec_layers", "dim_feedforward", "num_classes", "group_detr", "img_size")]


class InputDesc(ctypes.Structure):
    _fields_ = [("images", _vp), ("format", ctypes.c_int32), ("padding_mask", _vp), ("mean", ctypes.c_float * 3), ("std", ctypes.c_float * 3)]


IN_F32_NCHW, IN_16_NCHW, IN_U8_NHWC = 0, 1, 2
IMAGENET_MEAN, IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)      # demo/demo.py:150-153, datasets/coco.py


class FrameDesc(ctypes.Structure):
    """lwdetr_frame: one uint8 HWC RGB frame on the device, pixel (y, x) channel c at data + y*row_stride + x*3 + c."""
    _fields_ = [("data", _vp), ("height", ctypes.c_int32), ("width", ctypes.c_int32), ("row_stride", ctypes.c_int64)]


MAX_FRAMES, MAX_FRAME_SIDE = 1024, 8192      # LWDETR_MAX_FRAMES, LWDETR_MAX_FRAME_SIDE


class AuxOut(ctypes.Structure):
    _fields_ = [(n, _vp) for n in ("aux_logits", "aux_boxes", "enc_logits", "enc_boxes", "topk_index")]


def config_struct(cfg):
    c = ConfigStruct()
    c.vit_dim, c.vit_depth, c.vit_heads = cfg.vit_dim, cfg.vit_depth, cfg.vit_heads
    c.window_block_mask = sum(1 << i for i in cfg.window_blocks)
    taps = list(cfg.taps)
    c.n_taps = len(taps)
    for i, t in enumerate(taps):
        c.taps[i] = t
    c.n_levels = cfg.n_levels
    for i, p in enumerate(cfg.projector_scale):
        c.level_scale_log2[i] = {"P3": 1, "P4": 0, "P5": -1}[p]
    c.hidden_dim, c.sa_heads, c.ca_heads = cfg.hidden_dim, cfg.sa_nheads, cfg.ca_nheads
    c.dec_points, c.num_queries, c.dec_layers = cfg.dec_n_points, cfg.num_queries, cfg.dec_layers
    c.dim_feedforward, c.num_classes, c.group_detr, c.img_size = cfg.dim_feedforward, cfg.num_classes, cfg.group_detr, cfg.img_size
    return c


class Engine:
    """Owns one lwdetr_handle: packed weights + kernel schedule on the current CUDA device."""

    def __init__(self, cfg, dtype, device=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("lwdetr_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.cfg, self.dtype = cfg, dtype
        self._h = _vp()
        cs = config_struct(cfg)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        with torch.cuda.device(self.device):      # the handle binds to the device current at creation
            check(lib().lwdetr_create(ctypes.byref(cs), dtype_code(dtype), ctypes.byref(self._h)), "lwdetr_create")
        self._captures = []

    def close(self):
        if self._h:
            lib().lwdetr_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_state_dict(self, sd):
        """sd: name -> tensor with the reference state_dict names (any device/dtype; copied to CPU fp32)."""
        import torch
        names, keep = [], []
        for k, v in sd.items():
            if not torch.is_floating_point(v):
                continue                                    # num_batches_tracked
            names.append(k.encode())
            keep.append(v.detach().to("cpu", torch.float32).contiguous())
        n = len(names)
        c_names = (ctypes.c_char_p * n)(*names)
        c_ptrs = (_vp * n)(*[t.data_ptr() for t in keep])
        c_numel = (ctypes.c_int64 * n)(*[t.numel() for t in keep])
        check(lib().lwdetr_load_weights(self._h, n, ctypes.cast(c_names, _vp), ctypes.cast(c_ptrs, _vp),
                                        ctypes.cast(c_numel, _vp)), "lwdetr_load_weights")

    def broadcast_weights(self, nccl_comm, root=0):
        """One ncclBroadcast of the packed arena from rank `root` (nccl_comm: integer ncclComm_t, see b200/dist.py)."""
        check(lib().lwdetr_broadcast_weights(self._h, ctypes.c_void_p(nccl_comm), int(root), stream_ptr()), "lwdetr_broadcast_weights")

    def arena_bytes(self):
        return int(lib().lwdetr_weight_arena_bytes(self._h))

    def set_option(self, name, value):
        check(lib().lwdetr_set_option(self._h, name.encode(), int(value)), "lwdetr_set_option")

    def forward(self, images, want_aux=True, topk_override=None, mask=None, mean=IMAGENET_MEAN, std=IMAGENET_STD):
        """images: CUDA [B,3,R,R] fp32 / compute dtype, or CUDA uint8 [B,R,R,3] (HWC, normalised on the fly with mean/std),
        where R is cfg.img_size or a multiple of 64 in [448, 896] (config.input_resolution); mask: CUDA bool [B,R,R]
        (True = padded pixel) or None.  Returns the reference's output dict (fp32 CUDA tensors)."""
        import torch
        if images.device.type != "cuda":
            raise RuntimeError("lwdetr_b200: images must be CUDA tensors")
        if images.device != self.device:
            raise RuntimeError("lwdetr_b200: images are on %s but the engine lives on %s" % (images.device, self.device))
        hwc = images.dtype == torch.uint8
        S = int(images.shape[1 if hwc else 2]) if images.dim() == 4 else self.cfg.img_size
        if S != self.cfg.img_size and input_resolution(S, S, self.cfg.img_size) != S:
            raise RuntimeError("lwdetr_b200: input side %d is neither the configured %d nor a multiple of 64 in [%d, %d]"
                               % (S, self.cfg.img_size, MIN_IMG_SIZE, MAX_IMG_SIZE))
        desc = InputDesc()
        if hwc:
            if images.dim() != 4 or tuple(images.shape[1:]) != (S, S, 3):
                raise RuntimeError("lwdetr_b200: uint8 images must be [B, %d, %d, 3] (HWC), got %s" % (S, S, tuple(images.shape)))
            desc.format = IN_U8_NHWC
            for c in range(3):
                desc.mean[c], desc.std[c] = float(mean[c]), float(std[c])
        else:
            if images.dim() != 4 or images.shape[1] != 3 or images.shape[2] != S or images.shape[3] != S:
                raise RuntimeError("lwdetr_b200: expected images [B, 3, %d, %d], got %s" % (S, S, tuple(images.shape)))
            if images.dtype not in (torch.float32, self.dtype):
                images = images.float()
            desc.format = IN_F32_NCHW if images.dtype == torch.float32 else IN_16_NCHW
        images = images.contiguous()
        mk = None
        if mask is not None:
            if tuple(mask.shape) != (images.shape[0], S, S):
                raise RuntimeError("lwdetr_b200: mask must be [B, %d, %d], got %s" % (S, S, tuple(mask.shape)))
            mk = mask.to(device=self.device, dtype=torch.bool).contiguous()
        desc.images = images.data_ptr()
        desc.padding_mask = mk.data_ptr() if mk is not None else None
        B = images.shape[0]
        res, logits, boxes, aux = self._outputs(B, want_aux)
        ov = None
        if topk_override is not None:
            ov = topk_override.to(device=self.device, dtype=torch.int32).contiguous()
        check(lib().lwdetr_forward_at(self._h, ctypes.byref(desc), S, B, ptr(logits), ptr(boxes),
                                      ctypes.byref(aux) if aux is not None else None, ptr(ov), stream_ptr(self.device)), "lwdetr_forward_at")
        self._last_inputs = (images, ov, mk)    # keep alive until the stream has consumed them
        return res

    def forward_frames(self, frames, img_size=None, want_aux=True, mean=IMAGENET_MEAN, std=IMAGENET_STD, topk_override=None):
        """frames: CUDA uint8 RGB frames of any size - a [B, H, W, 3] tensor or a list of [H_i, W_i, 3] tensors, channel
        stride 1 and pixel stride 3, any row stride (cropped views are read in place).  Each frame is resized to
        img_size x img_size (default cfg.img_size) on the device exactly as Pillow's Image.resize((R, R), BILINEAR) -
        torchvision's Resize([R, R]) on a PIL image - then normalised with mean/std.  Returns forward()'s dict."""
        import torch
        R = self.cfg.img_size if img_size is None else int(img_size)
        if isinstance(frames, torch.Tensor):
            if frames.dim() != 4:
                raise RuntimeError("lwdetr_b200: frames must be [B, H, W, 3] or a list of [H, W, 3], got %s" % (tuple(frames.shape),))
            frames = list(frames.unbind(0))
        frames = list(frames)
        if not 1 <= len(frames) <= MAX_FRAMES:
            raise RuntimeError("lwdetr_b200: %d frames; a call takes 1 to %d" % (len(frames), MAX_FRAMES))
        descs = (FrameDesc * len(frames))()
        for i, f in enumerate(frames):
            if not isinstance(f, torch.Tensor) or f.dtype != torch.uint8:
                raise RuntimeError("lwdetr_b200: frame %d must be a uint8 tensor, got %s" % (i, getattr(f, "dtype", type(f))))
            if f.device != self.device:
                raise RuntimeError("lwdetr_b200: frame %d is on %s but the engine lives on %s" % (i, f.device, self.device))
            if f.dim() != 3 or f.shape[2] != 3:
                raise RuntimeError("lwdetr_b200: frame %d must be HWC RGB [H, W, 3], got %s" % (i, tuple(f.shape)))
            H, W = int(f.shape[0]), int(f.shape[1])
            if f.stride(2) != 1 or (W > 1 and f.stride(1) != 3):
                raise RuntimeError("lwdetr_b200: frame %d needs channel stride 1 and pixel stride 3, got strides %s" % (i, f.stride()))
            descs[i].data, descs[i].height, descs[i].width = f.data_ptr(), H, W
            descs[i].row_stride = f.stride(0) if H > 1 else 3 * W      # a one-row view may report any row stride
        m, s = (ctypes.c_float * 3)(*[float(v) for v in mean]), (ctypes.c_float * 3)(*[float(v) for v in std])
        B = len(frames)
        res, logits, boxes, aux = self._outputs(B, want_aux)
        ov = None
        if topk_override is not None:
            ov = topk_override.to(device=self.device, dtype=torch.int32).contiguous()
        check(lib().lwdetr_forward_frames(self._h, ctypes.cast(descs, _vp), B, R, ctypes.cast(m, _vp), ctypes.cast(s, _vp),
                                          ptr(logits), ptr(boxes), ctypes.byref(aux) if aux is not None else None, ptr(ov),
                                          stream_ptr(self.device)), "lwdetr_forward_frames")
        self._last_inputs = (frames, ov, None)   # keep alive until the stream has consumed them
        return res

    def _outputs(self, B, want_aux):
        """The result dict and the fp32 CUDA buffers the forward entry points write into."""
        import torch
        nq, nc, nl = self.cfg.num_queries, self.cfg.num_classes, self.cfg.dec_layers
        dev = self.device
        logits = torch.empty(B, nq, nc, device=dev, dtype=torch.float32)
        boxes = torch.empty(B, nq, 4, device=dev, dtype=torch.float32)
        aux = None
        res = {"pred_logits": logits, "pred_boxes": boxes}
        if want_aux:
            aux = AuxOut()
            al = torch.empty(nl - 1, B, nq, nc, device=dev, dtype=torch.float32)
            ab = torch.empty(nl - 1, B, nq, 4, device=dev, dtype=torch.float32)
            el = torch.empty(B, nq, nc, device=dev, dtype=torch.float32)
            eb = torch.empty(B, nq, 4, device=dev, dtype=torch.float32)
            ti = torch.empty(B, nq, device=dev, dtype=torch.int32)
            aux.aux_logits, aux.aux_boxes, aux.enc_logits, aux.enc_boxes, aux.topk_index = (
                al.data_ptr(), ab.data_ptr(), el.data_ptr(), eb.data_ptr(), ti.data_ptr())
            res["aux_outputs"] = [{"pred_logits": al[i], "pred_boxes": ab[i]} for i in range(nl - 1)]
            res["enc_outputs"] = {"pred_logits": el, "pred_boxes": eb}
            res["topk_index"] = ti
        return res, logits, boxes, aux

    # ---- debug captures -------------------------------------------------------------------------
    def capture(self, label, numel):
        import torch
        t = torch.empty(int(numel), dtype=torch.float32)
        check(lib().lwdetr_add_capture(self._h, label.encode(), ptr(t), int(numel)), "lwdetr_add_capture")
        self._captures.append((label, t))
        return t

    def capture_results(self):
        out = {}
        for i, (label, t) in enumerate(self._captures):
            n = lib().lwdetr_capture_result(self._h, i)
            out[label] = t[:n] if n >= 0 else None
        return out

    def clear_captures(self):
        lib().lwdetr_clear_captures(self._h)
        self._captures = []

    def ops(self):
        n = lib().lwdetr_num_ops(self._h)
        out = []
        for i in range(n):
            fl, by = ctypes.c_double(), ctypes.c_double()
            lib().lwdetr_op_cost(self._h, i, ctypes.byref(fl), ctypes.byref(by))
            out.append((lib().lwdetr_op_label(self._h, i).decode(), fl.value, by.value))
        return out

    def profile_ops(self, iters=10):
        n = lib().lwdetr_num_ops(self._h)
        ms = (ctypes.c_float * n)()
        check(lib().lwdetr_profile_ops(self._h, iters, ctypes.cast(ms, _vp), stream_ptr()), "lwdetr_profile_ops")
        return [(lab, fl, by, ms[i]) for i, (lab, fl, by) in enumerate(self.ops())]
