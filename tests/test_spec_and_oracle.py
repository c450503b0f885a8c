"""CPU tests: the state_dict table and the oracle are pinned to the reference.

Goldens (tests/golden/) were produced by tools/make_goldens.py running the UNMODIFIED reference."""
import json
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

from b200.config import CONFIGS, PARAMS_M  # noqa: E402
from b200.spec import num_parameters, param_spec  # noqa: E402
from b200.synth import synth_images, synth_state_dict  # noqa: E402
from oracle import lwdetr_oracle as orc  # noqa: E402

NAMES = ["tiny", "small", "medium", "large", "xlarge"]


def _sample(t, n=2048):
    f = t.detach().reshape(-1).float()
    step = max(1, f.numel() // n)
    return f[::step][:n].numpy()


@pytest.mark.parametrize("name", NAMES)
def test_state_dict_table_matches_reference(name):
    with open(os.path.join(GOLD, "state_dict_%s.json" % name)) as f:
        ref = {k: tuple(v) for k, v in json.load(f).items()}
    ours = {e.name: tuple(e.shape) for e in param_spec(CONFIGS[name])}
    assert ours == ref


@pytest.mark.parametrize("name", NAMES)
def test_param_count_matches_readme(name):
    # README.md:352-356 "Params (M)" column: a known-answer test of the factory wiring
    assert round(num_parameters(CONFIGS[name]) / 1e6, 1) == PARAMS_M[name]


@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_reference_goldens(name):
    g = np.load(os.path.join(GOLD, "ref_%s.npz" % name))
    B, wseed, iseed = [int(v) for v in g["meta"]]
    cfg = CONFIGS[name]
    sd = synth_state_dict(cfg, wseed)
    inter = {}
    out = orc.forward(sd, cfg, synth_images(B, iseed), inter=inter)

    def close(a, b, atol, what):
        err = np.abs(np.asarray(a) - np.asarray(b)).max()
        assert err <= atol, "%s: %g" % (what, err)

    close(out["pred_logits"], g["pred_logits"], 1e-4, "pred_logits")
    close(out["pred_boxes"], g["pred_boxes"], 1e-5, "pred_boxes")
    close(out["enc_outputs"]["pred_logits"], g["enc_logits"], 1e-4, "enc logits")
    close(out["enc_outputs"]["pred_boxes"], g["enc_boxes"], 1e-5, "enc boxes")
    for i, a in enumerate(out["aux_outputs"]):
        close(_sample(a["pred_logits"], 8192), g["aux%d_logits" % i], 1e-4, "aux logits")
        close(a["pred_boxes"], g["aux%d_boxes" % i], 1e-5, "aux boxes")
    for i in range(cfg.vit_depth):
        close(_sample(inter["block%d" % i]), g["block%d" % i], 1e-4, "block%d" % i)
    for l in range(cfg.n_levels):
        close(_sample(inter["level%d" % l]), g["level%d" % l], 2e-4, "level%d" % l)
    for i in range(cfg.dec_layers):
        close(_sample(inter["dec%d" % i]), g["dec%d" % i], 1e-4, "dec%d" % i)
    close(_sample(inter["query_pos"]), g["query_pos"], 1e-4, "query_pos")


def test_synthetic_weights_keep_activations_sane():
    cfg = CONFIGS["tiny"]
    inter = {}
    out = orc.forward(synth_state_dict(cfg, 1), cfg, synth_images(1, 0), inter=inter)
    for k in ("patch", "block5", "level0", "dec2"):
        assert 0.3 < inter[k].std().item() < 3.0 and inter[k].abs().max().item() < 60.0, k
    assert torch.isfinite(out["pred_logits"]).all() and torch.isfinite(out["pred_boxes"]).all()


def test_msda_core_matches_grid_sample_formulation():
    # the reference's own self-check recipe (models/ops/test.py:27-34,37-60): shapes/seed from there
    import torch.nn.functional as F
    torch.manual_seed(3)
    N, M, D, Lq, L, P = 1, 2, 2, 2, 2, 2
    shapes = [(6, 4), (3, 2)]
    S = sum(h * w for h, w in shapes)
    value = torch.rand(N, S, M, D, dtype=torch.float64) * 0.01
    loc = torch.rand(N, Lq, M, L, P, 2, dtype=torch.float64) * 1.4 - 0.2      # includes out-of-range points
    w = torch.rand(N, Lq, M, L, P, dtype=torch.float64) + 1e-5
    w = w / w.sum(-1, keepdim=True).sum(-2, keepdim=True)
    got = orc.msda_core(value, shapes, loc, w)
    # grid_sample restatement (ms_deform_attn_func.py:52-75)
    vals = value.split([h * w_ for h, w_ in shapes], dim=1)
    acc = []
    for l, (H, W) in enumerate(shapes):
        v = vals[l].flatten(2).transpose(1, 2).reshape(N * M, D, H, W)
        grid = (2 * loc[:, :, :, l] - 1).transpose(1, 2).flatten(0, 1)
        acc.append(F.grid_sample(v, grid, mode="bilinear", padding_mode="zeros", align_corners=False))
    aw = w.transpose(1, 2).reshape(N * M, 1, Lq, L * P)
    ref = (torch.stack(acc, dim=-2).flatten(-2) * aw).sum(-1).view(N, M * D, Lq).transpose(1, 2)
    assert torch.allclose(got, ref, rtol=1e-9, atol=1e-12)


def test_oracle_matches_live_reference_with_forced_topk():
    """The oracle against the reference's tiny forward on other weights and images than ref_tiny.npz
    (tests/golden/ref_tiny_seed5.npz, tools/make_goldens.py --live-only)."""
    g = np.load(os.path.join(GOLD, "ref_tiny_seed5.npz"))
    B, wseed, iseed = (int(v) for v in g["meta"])
    cfg = CONFIGS["tiny"]
    sd = synth_state_dict(cfg, wseed)
    x = synth_images(B, iseed)
    out = orc.forward(sd, cfg, x)
    assert (out["pred_logits"] - torch.from_numpy(g["pred_logits"])).abs().max().item() < 1e-4
    assert (out["pred_boxes"] - torch.from_numpy(g["pred_boxes"])).abs().max().item() < 1e-5


def test_reference_forward_export_is_the_last_layer_tuple():
    """SURVEY.md 8f-4, first half: after LWDETR.export() the reference's forward IS forward_export (lwdetr.py:103-109,
    176-195).  With the decoder in export mode only the last layer's hidden state is returned (transformer.py:406-414),
    so the tuple is (pred_boxes [B,nq,4], pred_logits [B,nq,C]) of the LAST decoder layer - bit-identical to the dict
    forward's pred_* on the same input.  This is the contract models.lwdetr.LWDETR.export() of the drop-in implements
    (checked against the device path in tests/test_model_gpu.py::test_export_tuple_equals_dict_outputs).  Both of the
    reference's outputs are stored in tests/golden/ref_tiny_seed5.npz (tools/make_goldens.py --live-only)."""
    g = np.load(os.path.join(GOLD, "ref_tiny_seed5.npz"))
    _, wseed, iseed = (int(v) for v in g["meta"])
    cfg = CONFIGS["tiny"]
    boxes, logits = torch.from_numpy(g["export_boxes"]), torch.from_numpy(g["export_logits"])
    assert boxes.shape == (1, cfg.num_queries, 4) and logits.shape == (1, cfg.num_queries, cfg.num_classes)
    assert torch.equal(boxes, torch.from_numpy(g["one_pred_boxes"])) and torch.equal(logits, torch.from_numpy(g["one_pred_logits"]))
    out = orc.forward(synth_state_dict(cfg, wseed), cfg, synth_images(1, iseed))
    assert (out["pred_logits"] - logits).abs().max().item() < 1e-4 and (out["pred_boxes"] - boxes).abs().max().item() < 1e-5


@pytest.mark.parametrize("name", ["tiny", "small", "medium", "large", "xlarge"])
def test_oracle_postprocess_matches_reference_golden(name):
    """oracle.postprocess == the reference's PostProcess.forward (lwdetr.py:515-544) run on the reference's own golden
    predictions (tests/golden/ref_postprocess.npz, made by tools/make_goldens.py --postprocess-only)."""
    g = np.load(os.path.join(GOLD, "ref_%s.npz" % name))
    p = np.load(os.path.join(GOLD, "ref_postprocess.npz"))
    out = {"pred_logits": torch.from_numpy(g["pred_logits"]), "pred_boxes": torch.from_numpy(g["pred_boxes"])}
    res = orc.postprocess(out, torch.from_numpy(p[name + "_sizes"]), int(p[name + "_num_select"][0]))
    assert int(p[name + "_num_select"][0]) == min(300, CONFIGS[name].num_queries)
    for b, r in enumerate(res):
        assert torch.equal(r["labels"], torch.from_numpy(p[name + "_labels"][b]))
        assert torch.equal(r["scores"], torch.from_numpy(p[name + "_scores"][b]))
        assert torch.allclose(r["boxes"], torch.from_numpy(p[name + "_boxes"][b]), rtol=0, atol=1e-4)


def test_oracle_padded_batch_matches_reference_golden():
    """Padded / mixed-size batch (NestedTensor.mask not all False): valid ratios, per-image proposals, memory and value
    masking of the oracle against the reference's own output (tests/golden/ref_tiny_padded.npz, tools/make_goldens.py
    --padded-only).  The device path still rejects such batches (SURVEY.md 8f rank 3); this pins the checker first."""
    g = np.load(os.path.join(GOLD, "ref_tiny_padded.npz"))
    cfg = CONFIGS["tiny"]
    B, wseed, iseed = (int(v) for v in g["meta"])
    x = synth_images(B, iseed).clone()
    mask = torch.zeros(B, 640, 640, dtype=torch.bool)
    for b, (h, w) in enumerate(g["valid"]):
        mask[b, int(h):, :] = True
        mask[b, :, int(w):] = True
        x[b][:, mask[b]] = 0
    sd = synth_state_dict(cfg, wseed)
    out = orc.forward(sd, cfg, x, mask=mask)
    assert (out["pred_logits"] - torch.from_numpy(g["pred_logits"])).abs().max().item() < 1e-4
    assert (out["pred_boxes"] - torch.from_numpy(g["pred_boxes"])).abs().max().item() < 1e-5
    assert (out["enc_outputs"]["pred_boxes"] - torch.from_numpy(g["enc_boxes"])).abs().max().item() < 1e-5
    # the masks matter: the same pixels without the mask give different predictions
    plain = orc.forward(sd, cfg, x)
    assert (plain["pred_logits"] - out["pred_logits"]).abs().max().item() > 1e-2
    # and an all-False mask is exactly the unpadded path
    same = orc.forward(sd, cfg, x, mask=torch.zeros_like(mask))
    assert torch.equal(same["pred_logits"], plain["pred_logits"])
