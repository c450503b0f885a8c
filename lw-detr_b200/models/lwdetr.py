"""B200-native LW-DETR module with the reference's `models.lwdetr` surface (lwdetr.py:36-216, 509-619):
LWDETR (an nn.Module whose parameters carry the reference's state_dict names), PostProcess, build().

The forward pass is NOT PyTorch: LWDETR.forward hands the image batch to the C-ABI engine
(include/lwdetr_b200.h, lwdetr_forward), which runs the hand-written sm_100a kernel schedule.  There is
no CPU / eager fallback: without the built library or without a CUDA device, forward raises."""
import os

import torch
from torch import nn

from b200 import capi
from b200.config import config_from_args, input_resolution
from b200.spec import param_spec
from util.misc import NestedTensor, nested_tensor_from_tensor_list

from ._tree import Holder, attach_entries
from .backbone import build_backbone


def _default_dtype():
    return {"bf16": torch.bfloat16, "fp16": torch.float16}[os.environ.get("LWDETR_B200_DTYPE", "fp16")]


class LWDETR(nn.Module):
    def __init__(self, cfg, backbone=None, aux_loss=True, compute_dtype=None):
        super().__init__()
        self.cfg = cfg
        self.num_queries = cfg.num_queries
        self.group_detr = cfg.group_detr
        self.aux_loss = aux_loss
        self.two_stage = True
        self.bbox_reparam = True
        self.lite_refpoint_refine = True
        self.compute_dtype = compute_dtype       # None: parameters' 16-bit dtype, else LWDETR_B200_DTYPE / fp16
        self.assume_frozen = False               # True: skip the per-forward weight-change check
        entries = [e for e in param_spec(cfg) if not e.name.startswith("backbone.0.")]
        attach_entries(self, entries)
        self.transformer.d_model = cfg.hidden_dim
        self.backbone = backbone if backbone is not None else build_backbone(None, cfg)
        self._export = False
        self._engine = None
        self._engine_sig = None

    # ------------------------------------------------------------------ engine management
    def _weights_signature(self):
        sig = []
        for t in list(self.parameters()) + list(self.buffers()):
            sig.append((t.data_ptr(), t._version, t.dtype, t.device))
        return hash(tuple(sig))

    def _resolve_dtype(self):
        if self.compute_dtype is not None:
            return self.compute_dtype
        p = self.class_embed.weight
        return p.dtype if p.dtype in (torch.float16, torch.bfloat16) else _default_dtype()

    def engine(self):
        """The packed CUDA engine for the current weights (re-packed when parameters change)."""
        dt = self._resolve_dtype()
        if self._engine is not None and self._engine.dtype == dt and (self.assume_frozen and self._engine_sig is not None):
            return self._engine
        sig = (self._weights_signature(), dt)
        pdev = next(self.parameters()).device
        if self._engine is None or self._engine.dtype != dt or (pdev.type == "cuda" and self._engine.device != pdev):
            if self._engine is not None:
                self._engine.close()
            self._engine = capi.Engine(self.cfg, dt, device=next(self.parameters()).device)
            self._engine_sig = None
        if self._engine_sig != sig:
            self._engine.load_state_dict(self.state_dict())
            self._engine_sig = sig
        return self._engine

    def __deepcopy__(self, memo):
        import copy
        new = LWDETR(self.cfg, aux_loss=self.aux_loss, compute_dtype=self.compute_dtype)
        new.load_state_dict(copy.deepcopy(self.state_dict(), memo))
        p = next(self.parameters())
        new.to(device=p.device, dtype=p.dtype)
        new.train(self.training)
        return new

    # ------------------------------------------------------------------ reference surface
    def export(self):
        self._export = True
        self.backbone.export()
        self.backbone[0].export()

    def update_drop_path(self, drop_path_rate, vit_encoder_num_layers):
        """Stochastic depth only acts in training (lwdetr.py:205-210); inference ignores it."""
        return None

    def update_dropout(self, drop_rate):
        return None

    @torch.no_grad()
    def forward(self, samples, targets=None):
        """samples: NestedTensor | list of [3,H,W] tensors | [B,3,H,W] tensor (lwdetr.py:111-127), or uint8 [B,R,R,3] frames.
        A square batch extent R that is a multiple of 64 in [448, 896] runs at R, as the reference does; any other extent
        up to cfg.img_size is padded to it with a padding mask (b200.config.input_resolution).
        Returns {'pred_logits' [B,nq,C], 'pred_boxes' [B,nq,4] (cxcywh, normalised), 'aux_outputs',
        'enc_outputs'} as fp32 CUDA tensors (lwdetr.py:161-174)."""
        if self.training:
            raise RuntimeError("lwdetr_b200 implements the inference forward only; call model.eval()")
        if isinstance(samples, torch.Tensor) and samples.dtype == torch.uint8:
            # raw camera / decoder frames [B, S, S, 3] (HWC, RGB, 0..255): the reference's host-side pre-processing
            # (demo.py:146-159: /255, Normalize(mean, std), HWC -> CHW) is fused into the patch-embed load on the device
            dev = next(self.parameters()).device
            if dev.type != "cuda":
                raise RuntimeError("lwdetr_b200: move the model to a CUDA device (no CPU fallback)")
            if samples.dim() == 4:
                self._check_export_size(input_resolution(samples.shape[1], samples.shape[2], self.cfg.img_size))
            out = self.engine().forward(samples.to(dev), want_aux=True)
            return self._pack_outputs(out)
        if isinstance(samples, (list, torch.Tensor)):
            samples = nested_tensor_from_tensor_list(samples)
        x, mask = samples.tensors, samples.mask
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("lwdetr_b200: move the model to a CUDA device (no CPU fallback)")
        if x.dim() != 4:
            raise RuntimeError("lwdetr_b200: expected a [B, 3, H, W] batch, got %s" % (tuple(x.shape),))
        S = input_resolution(x.shape[-2], x.shape[-1], self.cfg.img_size)
        self._check_export_size(S)
        if x.shape[-1] != S or x.shape[-2] != S:
            # a batch whose extent is not a native input size: pad to the configured size (bottom / right,
            # exactly what nested_tensor_from_tensor_list does between the images of a batch) and extend the mask
            xp = x.new_zeros((x.shape[0], x.shape[1], S, S))
            xp[:, :, : x.shape[-2], : x.shape[-1]] = x
            mp = torch.ones((x.shape[0], S, S), dtype=torch.bool, device=x.device)
            mp[:, : x.shape[-2], : x.shape[-1]] = mask if mask is not None else False
            x, mask = xp, mp
        x = x.to(dev)
        # the padding mask only matters when something IS padded (misc.py:317-339); an all-False mask takes the constant tables
        mask = mask.to(dev) if (mask is not None and bool(mask.any())) else None
        out = self.engine().forward(x, want_aux=True, mask=mask)
        return self._pack_outputs(out)

    @torch.no_grad()
    def forward_frames(self, frames, img_size=None):
        """frames: uint8 RGB frames of any size, as a decoder or camera delivers them - a [B, H, W, 3] tensor or a list of
        [H_i, W_i, 3] tensors (host tensors are moved to the model's device).  Each frame is resized to img_size x
        img_size (default cfg.img_size) on the device, bit-identical to the reference's host pre-processing
        (demo.py:146-159: transforms.Resize([R, R]) on a PIL image, ToTensor, Normalize), so the outputs equal
        forward() on those pre-processed images.  Boxes are normalised to each frame: PostProcess with target_sizes
        (H_i, W_i) gives them in source pixels."""
        if self.training:
            raise RuntimeError("lwdetr_b200 implements the inference forward only; call model.eval()")
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("lwdetr_b200: move the model to a CUDA device (no CPU fallback)")
        R = self.cfg.img_size if img_size is None else int(img_size)
        self._check_export_size(R)
        if isinstance(frames, torch.Tensor):
            frames = frames.to(dev)
        else:
            frames = [f.to(dev) if isinstance(f, torch.Tensor) else f for f in frames]
        return self._pack_outputs(self.engine().forward_frames(frames, img_size=R, want_aux=True))

    def _check_export_size(self, R):
        # the reference's forward_export adds pos_embed_export, computed once for the 40x40 grid (vit.py:328-332)
        if self._export and R != self.cfg.img_size:
            raise RuntimeError("lwdetr_b200: export mode runs at the configured %dx%d only, got %dx%d" % (self.cfg.img_size, self.cfg.img_size, R, R))

    def _pack_outputs(self, out):
        if self._export:
            return out["pred_boxes"], out["pred_logits"]      # forward_export tuple (lwdetr.py:176-195)
        res = {"pred_logits": out["pred_logits"], "pred_boxes": out["pred_boxes"]}
        if self.aux_loss:
            res["aux_outputs"] = out["aux_outputs"]
        res["enc_outputs"] = out["enc_outputs"]
        return res


class PostProcess(nn.Module):
    """lwdetr.py:509-544: sigmoid -> top `num_select` over (query, class) -> boxes to absolute xyxy."""

    def __init__(self, num_select=300):
        super().__init__()
        self.num_select = num_select

    @torch.no_grad()
    def forward(self, outputs, target_sizes):
        logits, boxes = outputs["pred_logits"], outputs["pred_boxes"]
        if len(logits) != len(target_sizes) or target_sizes.shape[1] != 2:
            raise ValueError("target_sizes must be [batch, 2]")
        ncls = logits.shape[2]
        if logits.is_cuda:
            # fused on the device (lwdetr_postprocess): only [B, num_select, 6] numbers are produced / leave the GPU
            scores, labels, xyxy = capi.postprocess(logits, boxes, target_sizes, self.num_select)
            labels = labels.long()
        else:
            # host tensors (e.g. outputs already copied to the CPU): plain torch, same arithmetic as the reference
            scores, flat = torch.topk(logits.sigmoid().flatten(1), self.num_select, dim=1)
            query, labels = flat // ncls, flat % ncls
            cx, cy, w, h = boxes.unbind(-1)
            xyxy = torch.stack([cx - 0.5 * w, cy - 0.5 * h, cx + 0.5 * w, cy + 0.5 * h], dim=-1)
            xyxy = torch.gather(xyxy, 1, query.unsqueeze(-1).expand(-1, -1, 4))
            img_h, img_w = target_sizes.unbind(1)
            xyxy = xyxy * torch.stack([img_w, img_h, img_w, img_h], dim=1)[:, None, :].to(xyxy.dtype)
        return [{"scores": s, "labels": l, "boxes": b} for s, l, b in zip(scores, labels, xyxy)]


class InferenceOnlyCriterion(nn.Module):
    """build() returns a criterion for API compatibility (lwdetr.py:596-619).  Losses / Hungarian matching
    are training-side and out of scope of the B200 inference path (SURVEY.md section 2)."""

    def __init__(self, weight_dict):
        super().__init__()
        self.weight_dict = weight_dict

    def forward(self, outputs, targets):
        raise NotImplementedError("lwdetr_b200 is an inference path: SetCriterion is not implemented")


def build(args):
    """(model, criterion, postprocessors) from the reference's argparse namespace (lwdetr.py:562-619)."""
    cfg = config_from_args(args)
    args.num_feature_levels = len(args.projector_scale)
    backbone = build_backbone(args, cfg)
    model = LWDETR(cfg, backbone=backbone, aux_loss=getattr(args, "aux_loss", True))
    weight_dict = {"loss_ce": getattr(args, "cls_loss_coef", 2), "loss_bbox": getattr(args, "bbox_loss_coef", 5),
                   "loss_giou": getattr(args, "giou_loss_coef", 2)}
    criterion = InferenceOnlyCriterion(weight_dict)
    postprocessors = {"bbox": PostProcess(num_select=getattr(args, "num_select", cfg.num_queries))}
    return model, criterion, postprocessors
