"""CPU tests of inference at square input sides other than 640: the oracle against the reference's own outputs at those
sizes (tests/golden/ref_res.npz, tools/make_goldens.py --resolution-only), the rule that maps a batch extent to the side
the model runs at, and the C-ABI declaration of the entry point that takes the side."""
import dataclasses
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

from b200.config import CONFIGS, MAX_IMG_SIZE, MIN_IMG_SIZE, input_resolution  # noqa: E402
from b200.synth import synth_images, synth_state_dict  # noqa: E402
from oracle import lwdetr_oracle as orc  # noqa: E402

RES_CASES = [("tiny", 448), ("small", 512), ("medium", 576), ("large", 768), ("xlarge", 896)]


def _sample(t, n=2048):
    f = t.detach().reshape(-1).float()
    step = max(1, f.numel() // n)
    return f[::step][:n].numpy()


def _close(a, b, atol, what):
    err = np.abs(np.asarray(a) - np.asarray(b)).max()
    assert err <= atol, "%s: %g" % (what, err)


def _check(g, case, cfg, out, inter):
    """Boxes are stored whole; logits and intermediates as strided samples whose length fixes the stride."""
    def sampled(t, key):
        return _sample(t, len(g[key]))

    _close(sampled(out["pred_logits"], case + "_pred_logits"), g[case + "_pred_logits"], 1e-4, "pred_logits")
    _close(out["pred_boxes"], g[case + "_pred_boxes"], 1e-5, "pred_boxes")
    _close(sampled(out["enc_outputs"]["pred_logits"], case + "_enc_logits"), g[case + "_enc_logits"], 1e-4, "enc logits")
    _close(out["enc_outputs"]["pred_boxes"], g[case + "_enc_boxes"], 1e-5, "enc boxes")
    for l in range(cfg.n_levels):
        _close(sampled(inter["level%d" % l], case + "_level%d" % l), g[case + "_level%d" % l], 2e-4, "level%d" % l)
    for i in range(cfg.dec_layers):
        _close(sampled(inter["dec%d" % i], case + "_dec%d" % i), g[case + "_dec%d" % i], 1e-4, "dec%d" % i)


@pytest.mark.parametrize("name,R", RES_CASES)
def test_oracle_matches_reference_at_other_resolutions(name, R):
    g = np.load(os.path.join(GOLD, "ref_res.npz"))
    case = "%s%d" % (name, R)
    B, wseed, iseed, size = (int(v) for v in g[case + "_meta"])
    assert size == R
    cfg = dataclasses.replace(CONFIGS[name], img_size=R)
    x = synth_images(B, iseed, R)
    inter = {}
    out = orc.forward(synth_state_dict(cfg, wseed), cfg, x, inter=inter)
    assert inter["tap0"].shape[1:3] == (R // 16, R // 16)
    _check(g, case, cfg, out, inter)


def res_padded_batch(g):
    """The padded fixture: images of the stored valid sizes, zero-padded to the stored square extent, and its mask."""
    B, _, iseed, extent = (int(v) for v in g["pad512_meta"])
    x = synth_images(B, iseed, extent).clone()
    mask = torch.zeros(B, extent, extent, dtype=torch.bool)
    for b, (h, w) in enumerate(g["pad512_valid"]):
        mask[b, int(h):, :] = True
        mask[b, :, int(w):] = True
        x[b][:, mask[b]] = 0
    return x, mask


def test_oracle_matches_reference_on_padded_batch_at_512():
    """A 512x512 and a 448x384 image batched together: the reference runs at the 512 extent with the padding mask."""
    g = np.load(os.path.join(GOLD, "ref_res.npz"))
    _, wseed, _, extent = (int(v) for v in g["pad512_meta"])
    assert input_resolution(extent, extent) == extent == 512
    cfg = dataclasses.replace(CONFIGS["tiny"], img_size=extent)
    x, mask = res_padded_batch(g)
    inter = {}
    out = orc.forward(synth_state_dict(cfg, wseed), cfg, x, inter=inter, mask=mask)
    _check(g, "pad512", cfg, out, inter)


@pytest.mark.parametrize("side", range(MIN_IMG_SIZE, MAX_IMG_SIZE + 1, 64))
def test_square_multiples_of_64_in_range_run_natively(side):
    assert input_resolution(side, side) == side
    assert input_resolution(side, side, img_size=640) == side


@pytest.mark.parametrize("hw", [(384, 384), (640, 576), (576, 640), (600, 600), (500, 500), (1, 1), (640, 640), (448, 512)])
def test_other_extents_up_to_640_are_padded_to_640(hw):
    assert input_resolution(*hw) == 640


@pytest.mark.parametrize("hw", [(960, 960), (700, 700), (704, 640), (896, 832), (960, 448), (1024, 1024)])
def test_other_extents_above_640_raise(hw):
    with pytest.raises(RuntimeError, match="larger than the configured 640x640"):
        input_resolution(*hw)


def test_header_declares_forward_at():
    with open(os.path.join(ROOT, "include", "lwdetr_b200.h")) as f:
        hdr = f.read()
    m = re.search(r"LWDETR_API\s+int\s+lwdetr_forward_at\s*\(([^;]*)\);", hdr)
    assert m, "lwdetr_forward_at is not declared"
    args = [a.strip() for a in m.group(1).split(",")]
    assert args[:3] == ["lwdetr_handle* h", "const lwdetr_input* input", "int img_size"]
    assert "#define LWDETR_MIN_IMG_SIZE %d" % MIN_IMG_SIZE in hdr and "#define LWDETR_MAX_IMG_SIZE %d" % MAX_IMG_SIZE in hdr
