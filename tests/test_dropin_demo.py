"""The reference's own caller, demo/demo.py, against the drop-in (SURVEY.md 8b, INTEGRATION.md 1): `from models import
build_model` resolves to this repo, and the model is built from exactly the namespace demo.py's argument parser yields for
the LW-DETR-small evaluation flags (tests/golden/demo_small_args.json, tools/make_goldens.py --live-only).  The steps
demo.main takes after that (load the checkpoint, resize to 640x640 and normalise, forward, PostProcess) run in a fresh
interpreter with only this repository on the path."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

DRIVER = r'''
import argparse, json, os, sys
import numpy as np
import torch
from PIL import Image
from torchvision import transforms
import models, util.misc
from models import build_model
from util.misc import nested_tensor_from_tensor_list
mode, args_json, weights, image, device = sys.argv[1:6]
with open(args_json) as f:
    args = argparse.Namespace(**json.load(f), weights=weights, input=image, device=device)
info = {"models_file": models.__file__, "has_nested_tensor": hasattr(util.misc, "NestedTensor")}
model, _, post = build_model(args)
model.to(torch.device("cpu" if mode == "build" else args.device)); model.eval()
ck = torch.load(args.weights, map_location="cpu")
model.load_state_dict(ck["model"], strict=True)
info["n_params"] = sum(p.numel() for p in model.parameters())
if mode == "build":
    try:
        model(nested_tensor_from_tensor_list([torch.zeros(3, 640, 640)]))
        info["cpu_forward"] = "ran"
    except RuntimeError as e:
        info["cpu_forward"] = str(e)
else:
    pil = Image.open(args.input).convert("RGB")
    x = transforms.Compose([transforms.Resize([640, 640]), transforms.ToTensor(),
                            transforms.Normalize([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])])(pil).to(args.device)
    sizes = torch.tensor([pil.size[::-1]], device=args.device)
    with torch.no_grad():
        pred = post["bbox"](model(nested_tensor_from_tensor_list([x])), sizes)[0]
    s, l, b = (pred[k].cpu() for k in ("scores", "labels", "boxes"))
    info.update({"n": len(s), "finite": bool(torch.isfinite(s).all() and torch.isfinite(b).all()),
                 "sorted": bool((s[:-1] >= s[1:]).all()), "labels_ok": bool(((l >= 0) & (l < 91)).all()),
                 "sizes": sizes.cpu().tolist()[0]})
print("RESULT " + json.dumps(info))
'''


def _run(mode, tmp_path, device):
    import numpy as np
    from PIL import Image
    sys.path.insert(0, os.path.join(ROOT, "lw-detr_b200"))
    from b200.config import CONFIGS
    from b200.synth import synth_state_dict
    ck = tmp_path / "small.pth"
    torch.save({"model": synth_state_dict(CONFIGS["small"], 1)}, ck)
    img = tmp_path / "in.jpg"
    rng = np.random.default_rng(0)
    Image.fromarray(rng.integers(0, 255, (427, 640, 3), dtype=np.uint8)).save(img)
    drv = tmp_path / "driver.py"
    drv.write_text(DRIVER)
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "lw-detr_b200"))
    cmd = [sys.executable, str(drv), mode, os.path.join(GOLD, "demo_small_args.json"), str(ck), str(img), device]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


def test_reference_demo_builds_and_loads_against_dropin(tmp_path):
    info = _run("build", tmp_path, "cpu")
    assert info["models_file"].startswith(os.path.join(ROOT, "lw-detr_b200"))      # the drop-in
    assert info["has_nested_tensor"]
    assert 14.0e6 < info["n_params"] < 17.0e6                                      # README.md:353 (14.6 M) + the 12 training-only query groups
    assert "no CPU fallback" in info["cpu_forward"] or "CUDA" in info["cpu_forward"]


@pytest.mark.gpu
def test_reference_demo_runs_end_to_end_on_the_gpu(tmp_path):
    info = _run("main", tmp_path, "cuda")
    assert info["n"] == 300 and info["finite"] and info["sorted"] and info["labels_ok"]      # --num_select 300
    assert info["sizes"] == [427, 640]
