"""Throughput, batch-1 latency and the heaviest kernels of one configuration at every square input side the reference
trains at (448 ... 896 in steps of 64), all through ONE engine handle (lwdetr_forward_at re-plans per side).

    python tools/bench_resolution.py --config small --batch 32 --dtype fp16 --out profiles/r03_resolution_small.json

Per side: images/s of the CUDA-graph forward at --batch on device-resident fp32 inputs (two alternating seeded batches,
CUDA events around --iters forwards after --warmup), p50 / p90 of --lat-iters single-image forwards (each timed with its
own events), and the five most expensive ops of lwdetr_profile_ops at --batch together with the window / global attention
totals and their achieved TFLOP/s.  The GPU's name and power limit are read by the same process and stored with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "lw-detr_b200"))

from b200 import capi  # noqa: E402
from b200.config import CONFIGS, MAX_IMG_SIZE, MIN_IMG_SIZE  # noqa: E402
from b200.synth import synth_images, synth_state_dict  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (r.stdout.strip().split(", ") + ["", "", ""])[:3] if r.returncode == 0 else ("", "", "")
    return {"name": name or torch.cuda.get_device_name(), "power_limit": power or "unavailable", "max_sm_clock": clock or "unavailable"}


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def measure(eng, R, batch, iters, warmup, lat_iters):
    dev = eng.device
    # batch-1 latency first: the throughput batch is planned last, so profile_ops below times that schedule
    x1 = synth_images(1, 7, R).to(dev)
    for _ in range(warmup):
        eng.forward(x1, want_aux=False)
    lat = []
    for _ in range(lat_iters):
        lat.append(events_ms(lambda i: eng.forward(x1, want_aux=False), 1))
    lat.sort()
    xs = [synth_images(batch, 100 + i, R).to(dev) for i in range(2)]
    for i in range(warmup):
        eng.forward(xs[i & 1], want_aux=False)
    ms = events_ms(lambda i: eng.forward(xs[i & 1], want_aux=False), iters)
    prof = eng.profile_ops(iters=10)
    top = sorted(prof, key=lambda r: -r[3])[:5]
    kinds = {}
    for lab, fl, _, t in prof:
        for kind in ("win_attn", "glb_attn"):
            if lab.endswith("." + kind):
                k = kinds.setdefault(kind, {"ms": 0.0, "flop": 0.0})
                k["ms"] += t
                k["flop"] += fl
    for k in kinds.values():
        k["tflops"] = k["flop"] / (k["ms"] * 1e-3) / 1e12 if k["ms"] > 0 else None
    return {
        "img_size": R, "tokens": (R // 16) ** 2, "window_tokens": (R // 64) ** 2,
        "images_per_s": batch * iters / (ms * 1e-3), "ms_per_batch": ms / iters,
        "latency_b1_ms_p50": lat[len(lat) // 2], "latency_b1_ms_p90": lat[int(len(lat) * 0.9)],
        "profile_ops_total_ms": sum(r[3] for r in prof),
        "top5_ops": [{"label": lab, "ms": t, "gflop": fl / 1e9} for lab, fl, _, t in top],
        "attention": kinds,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="small", choices=sorted(CONFIGS))
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--lat-iters", type=int, default=200)
    ap.add_argument("--sizes", default=",".join(str(r) for r in range(MIN_IMG_SIZE, MAX_IMG_SIZE + 1, 64)))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_resolution.py measures on a CUDA device; none is available")
    if a.iters < 50:
        raise SystemExit("--iters must be at least 50")
    cfg = CONFIGS[a.config]
    dt = {"fp16": torch.float16, "bf16": torch.bfloat16}[a.dtype]
    eng = capi.Engine(cfg, dt)
    eng.load_state_dict(synth_state_dict(cfg, 1))
    eng.set_option("cuda_graph", 1)
    rows = []
    for R in (int(s) for s in a.sizes.split(",")):
        rows.append(measure(eng, R, a.batch, a.iters, max(a.warmup, 2), a.lat_iters))
        print(json.dumps({k: v for k, v in rows[-1].items() if k != "top5_ops"}), flush=True)
    eng.close()
    rep = {"gpu": gpu_info(), "config": a.config, "dtype": a.dtype, "batch": a.batch, "iters": a.iters, "warmup": a.warmup,
           "lat_iters": a.lat_iters, "inputs": "device-resident fp32 [B,3,R,R], two alternating seeded batches, CUDA graph on",
           "torch": torch.__version__, "results": rows}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(rep, f, indent=1)
    print(json.dumps(rep["gpu"]))


if __name__ == "__main__":
    main()
