"""Cost of taking uint8 frames of any size (lwdetr_forward_frames: Pillow-exact resize fused into the patch gather) against
feeding frames that were already resized to the model's side (lwdetr_forward_at, uint8 [B,R,R,3]).

    python tools/bench_frames.py --config small --batch 32 --out profiles/r04_frames_small.json

One engine, CUDA graph on, all frames device-resident.  Per source size (720p, 1080p, 2160p):
  - images/s of forward_frames and of forward_at on the same frames pre-resized by Pillow, measured in alternating
    chunks of --iters forwards (CUDA events), --rounds times each; medians are reported;
  - the resize op's time from lwdetr_profile_ops (the "patch_gather" op, L2 not flushed), its bytes (source frames +
    patch matrix) and their share of the HBM bandwidth measured on B200 (6571.9 GB/s, DESIGN.md section 2);
  - per-frame Pillow resize time (transforms.Resize on a PIL image, one host core) - CPU time, for scale.
The GPU's name and power limit are read by the same process and stored with the numbers.
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch
from PIL import Image
from torchvision import transforms

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "lw-detr_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from b200 import capi  # noqa: E402
from b200.config import CONFIGS  # noqa: E402
from b200.synth import synth_state_dict  # noqa: E402
from bench_resolution import events_ms, gpu_info  # noqa: E402

HBM_GBS = 6571.9
SOURCES = {"720p": (720, 1280), "1080p": (1080, 1920), "2160p": (2160, 3840)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="small", choices=sorted(CONFIGS))
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_frames.py measures on a CUDA device; none is available")
    cfg = CONFIGS[a.config]
    R, B = cfg.img_size, a.batch
    dt = {"fp16": torch.float16, "bf16": torch.bfloat16}[a.dtype]
    eng = capi.Engine(cfg, dt)
    eng.load_state_dict(synth_state_dict(cfg, 1))
    eng.set_option("cuda_graph", 1)
    tf = transforms.Resize([R, R])
    rng = np.random.default_rng(0)
    rows = []
    for name, (H, W) in SOURCES.items():
        src = rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8)
        t0 = time.perf_counter()
        resized = np.stack([np.asarray(tf(Image.fromarray(f))) for f in src])
        pil_ms = (time.perf_counter() - t0) * 1e3 / B
        frames = torch.from_numpy(src).to(eng.device)
        pre = torch.from_numpy(resized).to(eng.device)
        del src, resized
        run_frames = lambda i: eng.forward_frames(frames, want_aux=False)   # noqa: E731
        run_at = lambda i: eng.forward(pre, want_aux=False)                 # noqa: E731
        for _ in range(a.warmup):
            run_at(0)
            run_frames(0)
        ips = {"frames": [], "at": []}
        for _ in range(a.rounds):
            ips["at"].append(B * a.iters / (events_ms(run_at, a.iters) * 1e-3))
            ips["frames"].append(B * a.iters / (events_ms(run_frames, a.iters) * 1e-3))
        run_frames(0)                       # the schedule's input op now reads these frames
        prof = {lab: (by, ms) for lab, _, by, ms in eng.profile_ops(iters=20)}
        by, ms = prof["patch_gather"]
        row = {
            "source": name, "height": H, "width": W,
            "forward_frames_images_per_s": statistics.median(ips["frames"]),
            "forward_at_preresized_images_per_s": statistics.median(ips["at"]),
            "rounds": {k: [round(v, 1) for v in vals] for k, vals in ips.items()},
            "resize_op_us": ms * 1e3, "resize_op_bytes": by, "resize_op_gbs": by / (ms * 1e-3) / 1e9,
            "resize_op_hbm_fraction": by / (ms * 1e-3) / 1e9 / HBM_GBS,
            "pillow_resize_ms_per_frame_cpu": pil_ms,
        }
        row["forward_frames_vs_at"] = row["forward_frames_images_per_s"] / row["forward_at_preresized_images_per_s"]
        rows.append(row)
        print(json.dumps({k: v for k, v in row.items() if k != "rounds"}), flush=True)
        del frames, pre
        torch.cuda.empty_cache()
    eng.close()
    rep = {"gpu": gpu_info(), "config": a.config, "dtype": a.dtype, "batch": B, "img_size": R, "iters": a.iters,
           "rounds": a.rounds, "hbm_gbs_reference": HBM_GBS, "cuda_graph": True,
           "inputs": "device-resident uint8 frames (seeded noise); forward_at gets the same frames resized by Pillow",
           "pillow_note": "CPU time on one host core of the GPU machine, torchvision Resize on a PIL image",
           "torch": torch.__version__, "results": rows}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(rep, f, indent=1)
    print(json.dumps(rep["gpu"]))


if __name__ == "__main__":
    main()
