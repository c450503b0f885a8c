"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference via
tools/ref_import.py) on the deterministic synthetic weights/inputs of b200/synth.py.

Run in the build container only:  python tools/make_goldens.py
Each fixture holds the reference's final outputs and strided samples of its intermediates (captured
with forward hooks), plus the state_dict names/shapes (tests/golden/state_dict_<cfg>.json).
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "lw-detr_b200"))

import ref_import  # noqa: E402
from b200.config import CONFIGS  # noqa: E402
from b200.synth import synth_images, synth_state_dict  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
CASES = [("tiny", 2), ("small", 1), ("medium", 1), ("large", 1), ("xlarge", 1)]
WEIGHT_SEED, IMAGE_SEED = 1, 0


def sample(t, n=2048):
    f = t.detach().reshape(-1).float()
    step = max(1, f.numel() // n)
    return f[::step][:n].numpy().copy()


POST_SIZES = [[480.0, 640.0], [640.0, 427.0]]     # (height, width) per image, as PostProcess takes them


def make_postprocess_goldens():
    """Reference PostProcess.forward (lwdetr.py:515-544) on the reference's own golden predictions: pins the oracle's
    postprocess() and, through it, the fused device kernel.  Only needs the existing ref_<cfg>.npz fixtures."""
    rec = {}
    for name, B in CASES:
        cfg = CONFIGS[name]
        _, _, post = ref_import.build_reference(cfg)
        gold = np.load(os.path.join(GOLD, "ref_%s.npz" % name))
        out = {"pred_logits": torch.from_numpy(gold["pred_logits"]), "pred_boxes": torch.from_numpy(gold["pred_boxes"])}
        sizes = torch.tensor(POST_SIZES[:B])
        with torch.no_grad():
            res = post["bbox"](out, sizes)
        rec[name + "_sizes"] = sizes.numpy()
        rec[name + "_num_select"] = np.array([post["bbox"].num_select], dtype=np.int64)
        rec[name + "_scores"] = torch.stack([r["scores"] for r in res]).numpy()
        rec[name + "_labels"] = torch.stack([r["labels"] for r in res]).numpy()
        rec[name + "_boxes"] = torch.stack([r["boxes"] for r in res]).numpy()
        print("postprocess", name, rec[name + "_scores"].shape, "num_select", post["bbox"].num_select)
    np.savez_compressed(os.path.join(GOLD, "ref_postprocess.npz"), **rec)


PAD_VALID = [(640, 640), (576, 480)]              # (valid height, valid width) of the two images of the padded fixture


def padded_inputs():
    """Two images of different size padded to 640x640 the way util/misc.py:317-339 builds a NestedTensor."""
    x = synth_images(2, 9).clone()
    mask = torch.zeros(2, 640, 640, dtype=torch.bool)
    for b, (h, w) in enumerate(PAD_VALID):
        mask[b, h:, :] = True
        mask[b, :, w:] = True
        x[b][:, mask[b]] = 0
    return x, mask


def make_padded_golden():
    """Reference forward on a padded / mixed-size batch (masks not all False): pins the oracle's valid-ratio,
    proposal-masking and value-masking arithmetic (SURVEY.md 8f rank 3) ahead of the device implementation."""
    cfg = CONFIGS["tiny"]
    model, _, _ = ref_import.build_reference(cfg)
    model.load_state_dict(synth_state_dict(cfg, 5), strict=True)
    x, mask = padded_inputs()
    nested = sys.modules["_ref_util.misc"].NestedTensor(x, mask)
    with torch.no_grad():
        out = model(nested)
    np.savez_compressed(os.path.join(GOLD, "ref_tiny_padded.npz"), pred_logits=out["pred_logits"].numpy(),
                        pred_boxes=out["pred_boxes"].numpy(), enc_boxes=out["enc_outputs"]["pred_boxes"].numpy(),
                        valid=np.array(PAD_VALID, dtype=np.int64), meta=np.array([2, 5, 9], dtype=np.int64))
    print("padded", out["pred_logits"].shape)


def make_live_goldens():
    """What the tests used to compute by running the reference next to them, stored so that they need no reference tree:
      ref_tiny_seed5.npz   the tiny forward on weight seed 5: dict outputs on two images (image seed 9), and on the first
                           image alone the dict outputs and the forward_export tuple after LWDETR.export()
      ref_msda_checker.npz models/ops/test.py's inputs (torch.manual_seed(3), double then float pass) and the output of
                           its checker ms_deform_attn_core_pytorch on them
      demo_small_args.json the namespace demo/demo.py's argument parser yields for the LW-DETR-small evaluation flags"""
    cfg = CONFIGS["tiny"]
    model, _, _ = ref_import.build_reference(cfg)
    model.load_state_dict(synth_state_dict(cfg, 5), strict=True)
    x1 = synth_images(1, 9)
    with torch.no_grad():
        two = model(synth_images(2, 9))
        one = model(x1)
        model.export()
        boxes, logits = model(x1)
    np.savez_compressed(os.path.join(GOLD, "ref_tiny_seed5.npz"), pred_logits=two["pred_logits"].numpy(),
                        pred_boxes=two["pred_boxes"].numpy(), one_pred_logits=one["pred_logits"].numpy(),
                        one_pred_boxes=one["pred_boxes"].numpy(), export_boxes=boxes.numpy(), export_logits=logits.numpy(),
                        meta=np.array([2, 5, 9], dtype=np.int64))

    ref_import._install_shims()
    ops = os.path.join(ref_import.REF, "models", "ops")
    sys.path.insert(0, ops)
    try:
        from functions.ms_deform_attn_func import ms_deform_attn_core_pytorch as core
    finally:
        sys.path.remove(ops)
    N, M, D, Lq, L, P = 1, 2, 2, 2, 2, 2                                   # models/ops/test.py:27-31
    shapes = torch.as_tensor([(6, 4), (3, 2)], dtype=torch.long)
    S = int(shapes.prod(1).sum())
    torch.manual_seed(3)
    rec = {"shapes": shapes.numpy()}
    for i, cast in enumerate((lambda t: t.double(), lambda t: t)):
        value = torch.rand(N, S, M, D) * 0.01
        loc = torch.rand(N, Lq, M, L, P, 2)
        aw = torch.rand(N, Lq, M, L, P) + 1e-5
        aw /= aw.sum(-1, keepdim=True).sum(-2, keepdim=True)
        rec.update({"value%d" % i: value.numpy(), "loc%d" % i: loc.numpy(), "aw%d" % i: aw.numpy(),
                    "out%d" % i: core(cast(value).permute(0, 2, 3, 1), shapes, cast(loc), cast(aw)).numpy()})
    np.savez_compressed(os.path.join(GOLD, "ref_msda_checker.npz"), **rec)

    import importlib.util
    sys.path.insert(0, ref_import.REF)
    try:
        spec = importlib.util.spec_from_file_location("ref_demo", os.path.join(ref_import.REF, "demo", "demo.py"))
        demo = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(demo)
        ns = demo.get_args_parser().parse_args(DEMO_SMALL_FLAGS + ["--weights", "-", "--input", "-"])
    finally:
        sys.path.remove(ref_import.REF)
    args = {k: v for k, v in vars(ns).items() if k not in ("weights", "input", "output_dir", "device")}
    with open(os.path.join(GOLD, "demo_small_args.json"), "w") as f:
        json.dump(args, f, indent=0, sort_keys=True)
    print("live goldens: tiny seed 5, MSDA checker, demo args (%d fields)" % len(args))


DEMO_SMALL_FLAGS = ("--encoder vit_tiny --vit_encoder_num_layers 10 --window_block_indexes 0 1 3 6 7 9 --out_feature_indexes 2 4 5 9 "
                    "--projector_scale P4 --hidden_dim 256 --sa_nheads 8 --ca_nheads 16 --dec_n_points 2 --dec_layers 3 --group_detr 13 "
                    "--two_stage --bbox_reparam --lite_refpoint_refine --num_select 300").split()     # scripts/lwdetr_small_coco_eval.sh:10-24


RES_CASES = [("tiny", 448, 2), ("small", 512, 1), ("medium", 576, 1), ("large", 768, 1), ("xlarge", 896, 1)]
RES_PAD_EXTENT, RES_PAD_VALID = 512, [(512, 512), (448, 384)]     # tiny, weight seed 1, image seed 9


def res_padded_inputs():
    """A 512x512 and a 448x384 image batched the way util/misc.py:317-339 does: padded to their common 512x512 extent."""
    x = synth_images(2, 9, RES_PAD_EXTENT).clone()
    mask = torch.zeros(2, RES_PAD_EXTENT, RES_PAD_EXTENT, dtype=torch.bool)
    for b, (h, w) in enumerate(RES_PAD_VALID):
        mask[b, h:, :] = True
        mask[b, :, w:] = True
        x[b][:, mask[b]] = 0
    return x, mask


# strided samples (sample()) keep the fixture small: logits and intermediates are sampled, boxes are stored whole.  A
# reader recovers the stride from the stored length: sample(t, len(stored)).
RES_LOGIT_SAMPLES, RES_ENC_LOGIT_SAMPLES, RES_FEATURE_SAMPLES = 2048, 1024, 512


def _run_with_samples(model, cfg, inp):
    """Reference forward: whole boxes, strided samples of the class logits and of level* / dec*."""
    rec, hooks = {}, []

    def proj_hook(m, a, o):
        for l, f in enumerate(o):
            rec["level%d" % l] = sample(f.flatten(2).transpose(1, 2), RES_FEATURE_SAMPLES)

    hooks.append(model.backbone[0].projector.register_forward_hook(proj_hook))
    for i, lay in enumerate(model.transformer.decoder.layers):
        hooks.append(lay.register_forward_hook(lambda m, a, o, i=i: rec.__setitem__("dec%d" % i, sample(o, RES_FEATURE_SAMPLES))))
    with torch.no_grad():
        out = model(inp)
    for h in hooks:
        h.remove()
    rec["pred_logits"] = sample(out["pred_logits"], RES_LOGIT_SAMPLES)
    rec["pred_boxes"] = out["pred_boxes"].numpy()
    rec["enc_logits"] = sample(out["enc_outputs"]["pred_logits"], RES_ENC_LOGIT_SAMPLES)
    rec["enc_boxes"] = out["enc_outputs"]["pred_boxes"].numpy()
    return rec


def make_resolution_golden():
    """ref_res.npz (about 0.2 MB): the reference at square input sizes other than 640 (its ViT resizes the position
    embedding to the token grid, vit.py:26-54, and everything downstream follows the feature map sizes).  Keys are
    '<case>_<field>' with
    case '<config><R>' for RES_CASES (weights seed 1, images seed 0) and 'pad512' for a padded tiny batch (weights
    seed 1, images seed 9); '<case>_meta' = [B, weight seed, image seed, R]."""
    rec = {}
    for name, R, B in RES_CASES:
        cfg = CONFIGS[name]
        model, _, _ = ref_import.build_reference(cfg)
        model.load_state_dict(synth_state_dict(cfg, WEIGHT_SEED), strict=True)
        case = "%s%d" % (name, R)
        for k, v in _run_with_samples(model, cfg, synth_images(B, IMAGE_SEED, R)).items():
            rec[case + "_" + k] = v
        rec[case + "_meta"] = np.array([B, WEIGHT_SEED, IMAGE_SEED, R], dtype=np.int64)
        print("resolution", case, rec[case + "_pred_boxes"].shape, flush=True)
    cfg = CONFIGS["tiny"]
    model, _, _ = ref_import.build_reference(cfg)
    model.load_state_dict(synth_state_dict(cfg, WEIGHT_SEED), strict=True)
    x, mask = res_padded_inputs()
    nested = sys.modules["_ref_util.misc"].NestedTensor(x, mask)
    for k, v in _run_with_samples(model, cfg, nested).items():
        rec["pad512_" + k] = v
    rec["pad512_meta"] = np.array([2, WEIGHT_SEED, 9, RES_PAD_EXTENT], dtype=np.int64)
    rec["pad512_valid"] = np.array(RES_PAD_VALID, dtype=np.int64)
    np.savez_compressed(os.path.join(GOLD, "ref_res.npz"), **rec)


def main():
    torch.set_num_threads(os.cpu_count())
    os.makedirs(GOLD, exist_ok=True)
    if "--resolution-only" in sys.argv:
        make_resolution_golden()
        return
    if "--postprocess-only" in sys.argv:
        make_postprocess_goldens()
        return
    if "--padded-only" in sys.argv:
        make_padded_golden()
        return
    if "--live-only" in sys.argv:
        make_live_goldens()
        return
    for name, B in CASES:
        cfg = CONFIGS[name]
        model, _, _ = ref_import.build_reference(cfg)
        with open(os.path.join(GOLD, "state_dict_%s.json" % name), "w") as f:
            json.dump({k: list(v.shape) for k, v in model.state_dict().items()}, f, indent=0, sort_keys=True)
        model.load_state_dict(synth_state_dict(cfg, WEIGHT_SEED), strict=True)
        x = synth_images(B, IMAGE_SEED)
        rec = {}
        hooks = []
        enc = model.backbone[0].encoder
        for i, blk in enumerate(enc.blocks):
            hooks.append(blk.register_forward_hook(lambda m, a, o, i=i: rec.__setitem__("block%d" % i, sample(o))))

        def proj_hook(m, a, o):
            for l, f in enumerate(o):
                rec["level%d" % l] = sample(f.flatten(2).transpose(1, 2))

        hooks.append(model.backbone[0].projector.register_forward_hook(proj_hook))
        for i, lay in enumerate(model.transformer.decoder.layers):
            hooks.append(lay.register_forward_hook(lambda m, a, o, i=i: rec.__setitem__("dec%d" % i, sample(o))))
        hooks.append(model.transformer.decoder.ref_point_head.register_forward_hook(
            lambda m, a, o: rec.__setitem__("query_pos", sample(o))))
        with torch.no_grad():
            out = model(x)
        for h in hooks:
            h.remove()
        rec["pred_logits"] = out["pred_logits"].numpy()
        rec["pred_boxes"] = out["pred_boxes"].numpy()
        rec["enc_logits"] = out["enc_outputs"]["pred_logits"].numpy()
        rec["enc_boxes"] = out["enc_outputs"]["pred_boxes"].numpy()
        for i, a in enumerate(out["aux_outputs"]):
            rec["aux%d_logits" % i] = sample(a["pred_logits"], 8192)
            rec["aux%d_boxes" % i] = a["pred_boxes"].numpy()
        rec["meta"] = np.array([B, WEIGHT_SEED, IMAGE_SEED], dtype=np.int64)
        np.savez_compressed(os.path.join(GOLD, "ref_%s.npz" % name), **rec)
        print(name, "B=%d" % B, {k: v.shape for k, v in rec.items() if k.startswith("pred")})
    make_postprocess_goldens()
    make_padded_golden()
    make_live_goldens()


if __name__ == "__main__":
    main()
