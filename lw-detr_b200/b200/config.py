"""The five released LW-DETR configurations (reference: scripts/lwdetr_{tiny,small,medium,large,xlarge}
_coco_eval.sh:9-25, models/backbone/backbone.py:46-53) and the mapping from the reference's argparse
namespace (main.py:39-183) to them."""
from dataclasses import dataclass, field
from typing import Tuple

_ENCODER_DIM = {"vit_tiny": 192, "vit_small": 384, "vit_base": 768}


@dataclass(frozen=True)
class LWDETRConfig:
    name: str
    encoder: str
    vit_depth: int
    window_blocks: Tuple[int, ...]
    out_feature_indexes: Tuple[int, ...]
    projector_scale: Tuple[str, ...]
    hidden_dim: int
    sa_nheads: int
    ca_nheads: int
    dec_n_points: int
    num_queries: int
    dec_layers: int = 3
    dim_feedforward: int = 2048
    group_detr: int = 13
    num_classes: int = 91
    vit_heads: int = 12
    img_size: int = 640
    patch: int = 16

    @property
    def vit_dim(self):
        return _ENCODER_DIM[self.encoder]

    @property
    def grid(self):
        return self.img_size // self.patch

    @property
    def tokens(self):
        return self.grid * self.grid

    @property
    def n_levels(self):
        return len(self.projector_scale)

    @property
    def level_shapes(self):
        f = {"P3": 2.0, "P4": 1.0, "P5": 0.5}
        return tuple((int(self.grid * f[p]), int(self.grid * f[p])) for p in self.projector_scale)

    @property
    def memory_len(self):
        return sum(h * w for h, w in self.level_shapes)

    @property
    def taps(self):
        return tuple(sorted(i if i >= 0 else i + self.vit_depth for i in self.out_feature_indexes))


# Square input sides the reference trains every released model at (datasets/coco.py:133,
# make_coco_transforms_square_div_64, selected by --square_resize_div_64 in every released script).
MIN_IMG_SIZE, MAX_IMG_SIZE = 448, 896


def input_resolution(height, width, img_size=640):
    """The side R at which a batch whose padded extent is height x width runs.

    A square extent whose side is a multiple of 64 in [MIN_IMG_SIZE, MAX_IMG_SIZE] runs natively (R = side): the reference
    ViT takes any token grid and resizes its position embedding to it (vit.py:26-54, 343-365), and the four windows per
    side stay whole.  Any other extent that fits into img_size x img_size is padded to it (bottom / right, with a padding
    mask), so R = img_size; anything else raises."""
    if height == width and height % 64 == 0 and MIN_IMG_SIZE <= height <= MAX_IMG_SIZE:
        return int(height)
    if height <= img_size and width <= img_size:
        return int(img_size)
    raise RuntimeError("lwdetr_b200: images larger than the configured %dx%d are not supported, got %dx%d (square sides that "
                       "are multiples of 64 in [%d, %d] run at their own size)" % (img_size, img_size, height, width,
                                                                                   MIN_IMG_SIZE, MAX_IMG_SIZE))


_W10 = (0, 1, 3, 6, 7, 9)
_T10 = (2, 4, 5, 9)
CONFIGS = {
    "tiny": LWDETRConfig("tiny", "vit_tiny", 6, (0, 2, 4), (1, 3, 5), ("P4",), 256, 8, 16, 2, 100),
    "small": LWDETRConfig("small", "vit_tiny", 10, _W10, _T10, ("P4",), 256, 8, 16, 2, 300),
    "medium": LWDETRConfig("medium", "vit_small", 10, _W10, _T10, ("P4",), 256, 8, 16, 2, 300),
    "large": LWDETRConfig("large", "vit_small", 10, _W10, _T10, ("P3", "P5"), 384, 12, 24, 4, 300),
    "xlarge": LWDETRConfig("xlarge", "vit_base", 10, _W10, _T10, ("P3", "P5"), 384, 12, 24, 4, 300),
}
PARAMS_M = {"tiny": 12.1, "small": 14.6, "medium": 28.2, "large": 46.8, "xlarge": 118.0}   # README.md:352-356


def config_from_args(args):
    """Build a config from the reference's argparse namespace (the fields lwdetr.py:562-619 reads)."""
    if args.encoder not in _ENCODER_DIM:
        raise NotImplementedError("lwdetr_b200 supports the ViT encoders only, got %r" % (args.encoder,))
    for flag in ("two_stage", "bbox_reparam", "lite_refpoint_refine"):
        if not getattr(args, flag, False):
            raise NotImplementedError("lwdetr_b200 implements the released configuration (--%s)" % flag)
    scales = tuple(args.projector_scale)
    if scales not in (("P4",), ("P3", "P5")):
        raise NotImplementedError("projector_scale %r is not one of the released configurations" % (scales,))
    num_classes = 91 if args.dataset_file == "coco" else (366 if args.dataset_file == "o365" else 20)
    return LWDETRConfig(
        name="custom", encoder=args.encoder, vit_depth=int(args.vit_encoder_num_layers),
        window_blocks=tuple(args.window_block_indexes), out_feature_indexes=tuple(args.out_feature_indexes),
        projector_scale=scales, hidden_dim=int(args.hidden_dim), sa_nheads=int(args.sa_nheads),
        ca_nheads=int(args.ca_nheads), dec_n_points=int(args.dec_n_points), num_queries=int(args.num_queries),
        dec_layers=int(args.dec_layers), dim_feedforward=int(args.dim_feedforward),
        group_detr=int(args.group_detr), num_classes=num_classes)
