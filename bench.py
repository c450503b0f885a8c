"""LW-DETR inference throughput benchmark (BASELINE.json: images/sec at 640x640, per-GPU batch, N B200s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config small] [--batch 32] [--dtype fp16]
    python bench.py --impl reference ...      # the unmodified reference's CPU forward (baseline/_ref) on the host cores
    python bench.py --dump-outputs DIR ...    # also write the last timed step's predictions as DIR/<name>.npy
    torchrun --nproc-per-node N bench.py --gpus N ...   # one process per GPU, image-sharded replicas

One "step" = one forward pass of `batch` synthetic 640x640 images per GPU through the C-ABI engine
(random-init weights of the named architecture, b200/synth.py).  `value` = images/s of the whole job
with the inputs resident in HBM; `e2e` = the same through the public nn.Module call with PINNED HOST
inputs (H2D of every batch and D2H of the predictions inside the timed region, double buffered).
Rank 0 prints ONE JSON line.

With --dump-outputs DIR rank 0 writes what the last timed step returned to its caller, pred_logits [batch, queries,
classes] and pred_boxes [batch, queries, 4], as float32 DIR/pred_logits.npy and DIR/pred_boxes.npy.  Weights and inputs
are seeded, so two builds run with the same arguments can be compared output for output.  When the two arrays would
exceed 64 MB, a fixed seeded sample of the images is written instead, with its image indices in DIR/image_index.npy.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "lw-detr_b200"))

import torch  # noqa: E402

DUMP_LIMIT_BYTES = 63_000_000        # --dump-outputs stays under 64 MB, .npy headers and the image index included
DEFAULT_BATCH = {"tiny": 32, "small": 32, "medium": 64, "large": 32, "xlarge": 16}
FLOPS_PER_IMAGE = {"tiny": 21.40e9, "small": 31.76e9, "medium": 83.93e9, "large": 137.51e9, "xlarge": 342.51e9}  # SURVEY.md 8


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p.update({k: m[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in m})
        p["source"] = "measured"
    except Exception:
        pass
    return p


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons of one GPU with nvidia-smi while the timed region runs."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop = index, [], threading.Event()

    def run(self):
        try:
            p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        self.proc = p
        for line in p.stdout:
            self.rows.append([time.time()] + [c.strip() for c in line.split(",")])
            if self._stop.is_set():
                break
        try:
            p.kill()
        except Exception:
            pass

    def stop(self):
        self._stop.set()
        try:
            self.proc.kill()
        except Exception:
            pass

    def count_in(self, t0, t1):
        return sum(1 for r in self.rows if t0 <= r[0] <= t1)

    def summary(self, t0=0.0, t1=float("inf")):
        """Median SM clock / throttle reasons over the samples taken while the GPU was under bench load."""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if not (t0 <= r[0] <= t1):
                continue
            r = r[1:]
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        hot = [v for v in sm if v >= 0.5 * max(sm)]      # samples taken between two launches read an idle clock
        return {"sm_mhz": statistics.median(hot), "sm_mhz_unfiltered_median": statistics.median(sm), "sm_mhz_min": min(sm),
                "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm), "samples_kept": len(hot)}


def cpu_reference_run(cfg_name, steps, warmup, sample_batch, dtype_name, full_batch=0, budget_s=0.0):
    """The reference's CPU forward on the host cores, fp32, all the threads that help.
    kind "reference": the UNMODIFIED reference model built by its own models.build_model(args) (tools/ref_import.py;
    /root/reference in the build container, the byte-identical copy under baseline/_ref on the GPU box, staged by
    tools/vendor_reference.py at build() time), cross-attention through its ms_deform_attn_core_pytorch path - the path
    the reference itself takes on the CPU.  kind "port": the oracle port (oracle/lwdetr_oracle.py), only when no
    reference tree is available."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from b200.config import CONFIGS
    from b200.synth import synth_images, synth_state_dict
    cfg = CONFIGS[cfg_name]
    sd = synth_state_dict(cfg, 1)
    x = synth_images(sample_batch, 0)
    kind, fwd = "port", None
    try:
        import ref_import
        if ref_import.available():
            model, _, _ = ref_import.build_reference(cfg)
            model.load_state_dict(sd, strict=True)

            def fwd():
                with torch.no_grad():
                    return model(x)
            kind = "reference"
    except Exception as ex:   # a broken copy must not take the bench line down: fall back to the port and say so
        sys.stderr.write("reference import failed (%r): timing the oracle port instead\n" % (ex,))
        fwd = None
    if fwd is None:
        from oracle import lwdetr_oracle as orc
        fwd = lambda: orc.forward(sd, cfg, x)
    # "all the host threads it can use": torch's intra-op pool does not scale to every core of a many-core host
    # on ops this small, so pick the thread count that maximises throughput (one probe forward per candidate).
    ncpu = os.cpu_count() or 1
    best_t, best = ncpu, None
    for t in sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(t)
        fwd()
        t0 = time.perf_counter()
        fwd()
        el = time.perf_counter() - t0
        if best is None or el < best:
            best, best_t = el, t
    torch.set_num_threads(best_t)
    # One step = `per_step` images = per_step / sample_batch chunked forwards.  With a time budget the step is the full
    # per-GPU batch when (steps + warmup) of those fit, else the largest multiple of the chunk that does.
    chunks = 1
    if full_batch and budget_s > 0:
        t_chunk = best
        fit = int(budget_s / max(1e-9, (steps + warmup) * t_chunk))
        chunks = max(1, min(full_batch // sample_batch, fit))
    for _ in range(warmup * chunks):
        fwd()
    t0 = time.perf_counter()
    for _ in range(steps * chunks):
        fwd()
    dt = time.perf_counter() - t0
    per_step = sample_batch * chunks
    what = "unmodified reference models.build_model forward (baseline/_ref)" if kind == "reference" else "fp32 torch CPU oracle port"
    return {"value": steps * per_step / dt, "unit": "images/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": "%d step(s) of %d synthetic 640x640 image(s) each (%d forward(s) of %d), LW-DETR-%s, fp32, %s, best of thread counts up to %d"
                      % (steps, per_step, chunks, sample_batch, cfg_name, what, ncpu),
            "ms_per_step": 1e3 * dt / steps, "images_per_step": per_step}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="small")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step")
    ap.add_argument("--dtype", default=None, choices=[None, "fp16", "bf16"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-pdl", action="store_true", help="disable programmatic dependent launch (A/B measurements)")
    ap.add_argument("--profile-out", default=None, help="write the per-op timing table (JSON) here")
    ap.add_argument("--no-per-config", action="store_true", help="skip the per_config block (the other four BASELINE configs, N = 1 only)")
    ap.add_argument("--e2e-input", default="uint8", choices=["uint8", "fp32"], help="what the end-to-end arm holds on the host")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="write the last timed step's predictions to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cfg_name = a.config
    batch = a.batch or DEFAULT_BATCH[cfg_name]
    dtype_name = a.dtype or ("bf16" if cfg_name == "medium" else "fp16")
    warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    base_cfg = {"workload": "LW-DETR-%s forward, batch %d/GPU, 640x640 synthetic, random-init weights" % (cfg_name, batch),
                "per_gpu_batch": batch, "global_batch": batch * max(world, 1), "parallelism": "image-sharded replicas x%d" % max(world, 1)}

    if a.impl == "reference":
        if rank != 0:
            return
        # a bounded sample of the workload: the CPU forward is per-image independent, so images/s on a batch of
        # `sample` images is the same metric; the batch the reference arm ACTUALLY ran is what config states
        chunk = 4 if cfg_name in ("tiny", "small") else 2
        r = cpu_reference_run(cfg_name, max(1, a.steps), a.warmup, chunk, dtype_name, full_batch=batch, budget_s=240.0)
        if r["images_per_step"] != batch:
            # the bounded sample is smaller than the GPU arm's step: say what was run, not what the GPU arm runs
            base_cfg = dict(base_cfg)
            base_cfg.update({"workload": "LW-DETR-%s forward on the host CPU, %d images per step (bounded sample of the batch-%d/GPU workload; the forward is "
                                         "per-image independent), 640x640 synthetic, random-init weights" % (cfg_name, r["images_per_step"], batch),
                             "per_gpu_batch": r["images_per_step"], "global_batch": r["images_per_step"], "gpu_workload_batch": batch})
        print(json.dumps({
            "impl": "reference", "metric": "images/sec (640x640)", "value": r["value"], "unit": "images/s", "n_gpus": a.gpus,
            "steps": max(1, a.steps), "warmup": a.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": base_cfg,
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return

    # ------------------------------------------------------------------------------------ our arm
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    r = measure_config(cfg_name, batch, dtype_name, a.steps, warmup, dev, rank, world, local, graph=not a.no_graph, pdl=not a.no_pdl,
                       profile_out=a.profile_out, clocks=True, e2e_input=a.e2e_input, dump_dir=a.dump_outputs if rank == 0 else None)

    cpu = None
    if rank == 0 and world == 1:
        try:
            cpu = cpu_reference_run(cfg_name, 2, 1, 4 if cfg_name in ("tiny", "small") else 2, dtype_name)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as ex:
            cpu = {"error": repr(ex)}

    # ---- the other BASELINE configurations, measured in the same run (N = 1 only; a few seconds each): the bench line of
    # the headline config stays the contract, this block is the driver-visible evidence for the rest of the model family
    per_config = None
    if rank == 0 and world == 1 and not a.no_per_config:
        per_config = {}
        for name in ("tiny", "medium", "large", "xlarge"):
            if name == cfg_name:
                continue
            try:
                dn = "bf16" if name == "medium" else "fp16"
                q = measure_config(name, DEFAULT_BATCH[name], dn, max(5, a.steps // 2), 3, dev, 0, 1, local, graph=not a.no_graph, pdl=not a.no_pdl,
                                   profile_out=None, clocks=False, e2e_input=a.e2e_input)
                ro = q["roofline"] or {}
                per_config[name] = {"batch": DEFAULT_BATCH[name], "dtype": dn, "images_per_s": q["value"], "ms_per_step": q["ms_per_step"],
                                    "e2e_images_per_s": q["e2e"]["value"], "p50_latency_bs1_ms": q["p50_latency_bs1_ms"],
                                    "dominant_kernel": ro.get("kernel"), "dominant_share_of_step": ro.get("share_of_step"),
                                    "dominant_bound": ro.get("bound"), "dominant_frac": ro.get("frac"),
                                    "dominant_exp_frac": (ro.get("exp_bound") or {}).get("frac"),
                                    "whole_model_tensor_frac_of_sustained": q["whole_model_tensor_frac_of_sustained"]}
            except Exception as ex:
                per_config[name] = {"error": repr(ex)}

    if rank == 0:
        cfgd = dict(base_cfg)
        cfgd.update(r["config_extra"])
        print(json.dumps({
            "metric": "images/sec (640x640)", "value": r["value"], "unit": "images/s", "n_gpus": world, "steps": a.steps, "warmup": warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype_name,
            "data": "synthetic", "config": cfgd, "clocks": r["clocks"], "e2e": r["e2e"],
            "gpu_launches": r["n_kernels"] * a.steps, "p50_latency_bs1_ms": r["p50_latency_bs1_ms"],
            "p50_latency_bs1_e2e_postprocess_ms": r["p50_latency_bs1_e2e_postprocess_ms"], "roofline": r["roofline"], "cpu_baseline": cpu,
            "top_ops": r["top_ops"], "per_config": per_config}))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out, dump_dir):
    """Writes the predictions of one step as float32 .npy files (see the module docstring)."""
    import numpy as np
    arrays = {k: out[k].detach().float().cpu() for k in ("pred_logits", "pred_boxes")}
    batch = arrays["pred_logits"].shape[0]
    per_image = sum(v[0].numel() * 4 for v in arrays.values())
    keep = min(batch, DUMP_LIMIT_BYTES // (per_image + 8))
    os.makedirs(dump_dir, exist_ok=True)
    if keep < batch:
        idx = torch.randperm(batch, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["image_index"] = idx.double()
    for k, v in arrays.items():
        np.save(os.path.join(dump_dir, k + ".npy"), v.numpy())


def measure_config(cfg_name, batch, dtype_name, steps, warmup, dev, rank, world, local, graph=True, pdl=True, profile_out=None, clocks=True,
                   e2e_input="uint8", dump_dir=None):
    """One LW-DETR configuration on this rank's GPU: device-resident throughput, end-to-end throughput through the public
    module call with host inputs, batch-1 latencies and the per-kernel table.  Returns a dict (see main).  With dump_dir the
    predictions of the last timed step are written there (dump_outputs)."""
    import torch.distributed as dist
    from b200.config import CONFIGS
    from b200.synth import synth_images, synth_state_dict
    from models.lwdetr import LWDETR
    cfg = CONFIGS[cfg_name]
    dt = {"fp16": torch.float16, "bf16": torch.bfloat16}[dtype_name]
    # weights: rank 0 holds the real ones, every other rank packs DIFFERENT (seeded by its rank) weights of the same shapes -
    # that only fixes the arena layout - and ONE ncclBroadcast of the packed arena through the C ABI
    # (lwdetr_broadcast_weights, SURVEY.md 8e) makes them rank 0's.  No other collective touches the data path.
    model = LWDETR(cfg, compute_dtype=dt).eval()
    model.load_state_dict(synth_state_dict(cfg, 1 if rank == 0 else 1000 + rank), strict=True)
    model.to(dev)
    eng = model.engine()
    model.assume_frozen = True
    bcast_bytes, replicas_agree = 0, None
    if world > 1:
        from b200.dist import broadcast_engine_weights
        bcast_bytes = broadcast_engine_weights(eng, dev, src=0)
        probe = eng.forward(synth_images(1, seed=12345).to(dev), want_aux=False)
        sig = torch.stack([probe["pred_logits"].double().sum(), probe["pred_boxes"].double().sum()])
        allsig = [torch.empty_like(sig) for _ in range(world)]
        dist.all_gather(allsig, sig)
        replicas_agree = bool(all(torch.equal(s_, allsig[0]) for s_ in allsig))     # bit-identical replicas after the broadcast
    eng.set_option("cuda_graph", 1 if graph else 0)
    eng.set_option("pdl", 1 if pdl else 0)
    # inputs: two distinct device batches (fp32, 4.9 MB/image => larger than the 126 MB L2 at batch >= 26)
    xs = [synth_images(batch, seed=100 * rank + i).to(dev) for i in range(2)]
    in_bytes = xs[0].numel() * 4

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return ms.item()

    last = {}

    def dev_step(i):
        last["out"] = eng.forward(xs[i & 1], want_aux=False)
    for i in range(warmup):
        dev_step(i)
    sampler = ClockSampler(local)
    if rank == 0 and clocks:
        sampler.start()
        time.sleep(0.3)
    load_t0 = time.time()
    ms_total = timed(dev_step, steps)
    load_t1 = time.time()
    if dump_dir:
        dump_outputs(last["out"], dump_dir)       # before any untimed step below replaces it
    if rank == 0 and clocks:
        # a short timed region can fall between two 100 ms nvidia-smi samples: keep the same step running
        # (untimed) until at least three samples were taken under this load
        while sampler.count_in(load_t0 + 0.05, load_t1) < 3 and time.time() - load_t0 < 4.0 and sampler.is_alive():
            for i in range(4):
                dev_step(i)
            torch.cuda.synchronize()
            load_t1 = time.time()
        sampler.stop()
    value = world * batch * steps / (ms_total * 1e-3)

    # ---- end to end through the public module call: what a caller holds on the HOST (pinned) -> device (double buffered)
    # -> predictions back on the host.  "uint8": decoded frames [B, 640, 640, 3] as demo.py:146-159 holds them before its
    # host-side ToTensor / Normalize - that pre-processing is fused into the patch-embed load on the device (SURVEY.md 8f-2);
    # "fp32": the reference's own input contract, already normalised [B, 3, 640, 640] fp32 tensors.
    S = cfg.img_size
    hl = [torch.empty(batch, cfg.num_queries, cfg.num_classes, dtype=torch.float32).pin_memory() for _ in range(2)]
    hb = [torch.empty(batch, cfg.num_queries, 4, dtype=torch.float32).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)

    def e2e_measure(kind, d2h_stream=None):
        g = torch.Generator().manual_seed(7 + rank)
        if kind == "uint8":
            host = [torch.randint(0, 256, (batch, S, S, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
        else:
            host = [synth_images(batch, seed=7 + i).pin_memory() for i in range(2)]
        dbuf = [torch.empty_like(host[0], device=dev) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]

        def upload(i):
            s_ = i & 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[s_])
                dbuf[s_].copy_(host[s_], non_blocking=True)
                ready[s_].record(copy_stream)

        def run(n):
            for s_ in range(2):
                freed[s_].record(main_stream)
            upload(0)
            for i in range(n):
                s_ = i & 1
                if i + 1 < n:
                    upload(i + 1)
                main_stream.wait_event(ready[s_])
                out = model(dbuf[s_])
                freed[s_].record(main_stream)
                if d2h_stream is None:
                    hl[s_].copy_(out["pred_logits"], non_blocking=True)
                    hb[s_].copy_(out["pred_boxes"], non_blocking=True)
                else:
                    # read-back on its own stream: the next forward does not queue behind it (every forward writes freshly
                    # allocated output tensors, so nothing is overwritten while the copy runs)
                    d2h_stream.wait_stream(main_stream)
                    with torch.cuda.stream(d2h_stream):
                        hl[s_].copy_(out["pred_logits"], non_blocking=True)
                        hb[s_].copy_(out["pred_boxes"], non_blocking=True)
                    out["pred_logits"].record_stream(d2h_stream)
                    out["pred_boxes"].record_stream(d2h_stream)
            if d2h_stream is not None:
                main_stream.wait_stream(d2h_stream)                # the timed region ends when the last read-back has landed
        run(6)                                             # warm-up: also lets the caching allocator reach its steady state (outputs are freed a stream event later)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(steps)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return world * batch * steps / (ms.item() * 1e-3), host[0].numel() * host[0].element_size()

    d2h = hl[0].numel() * 4 + hb[0].numel() * 4
    d2h_stream = torch.cuda.Stream(device=dev)         # read-back on its own stream: +3 % end to end in a same-process A/B on the B200
    e2e_value, h2d = e2e_measure(e2e_input, d2h_stream)
    other = "fp32" if e2e_input == "uint8" else "uint8"
    e2e_other, h2d_other = e2e_measure(other, d2h_stream)
    if os.environ.get("LWDETR_BENCH_E2E_AB"):          # development aid: same-process A/B of the read-back placement
        st2 = torch.cuda.Stream(device=dev)
        for _ in range(3):
            sys.stderr.write("e2e A/B (%s): same stream %.1f | own stream %.1f images/s\n"
                             % (e2e_input, e2e_measure(e2e_input)[0], e2e_measure(e2e_input, st2)[0]))
    e2e = {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "host_input": e2e_input,
           "note": "public LWDETR module call; pinned host %s images (%s), double-buffered H2D on a copy stream, predictions copied to pinned host on a third stream"
                   % (e2e_input, "[B,640,640,3] raw frames, /255 + Normalize fused on the device" if e2e_input == "uint8" else "[B,3,640,640] normalised"),
           "with_%s_host_input" % other: {"value": e2e_other, "h2d_bytes_per_step": h2d_other}}

    # ---- p50 latency at batch 1 (CUDA graph), per GPU
    lat = None
    try:
        x1 = synth_images(1, seed=3).to(dev)
        for _ in range(5):
            eng.forward(x1, want_aux=False)
        torch.cuda.synchronize()
        ts = []
        for _ in range(50):
            t0 = time.perf_counter()
            eng.forward(x1, want_aux=False)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        lat = statistics.median(ts)
    except Exception as ex:  # noqa
        lat = None

    # ---- end-to-end p50 at batch 1 through the public surface: pinned host frame -> H2D -> LWDETR module -> fused
    # PostProcess on the device -> [num_select, 6] numbers back on the host (what demo.py does per image)
    lat_e2e = None
    try:
        from models.lwdetr import PostProcess
        post = PostProcess(num_select=min(300, cfg.num_queries))
        if e2e_input == "uint8":
            h1 = torch.randint(0, 256, (1, S, S, 3), dtype=torch.uint8).pin_memory()
        else:
            h1 = synth_images(1, seed=5).pin_memory()
        d1 = torch.empty_like(h1, device=dev)
        sizes = torch.tensor([[640.0, 640.0]], device=dev)
        ts = []
        for i in range(60):
            t0 = time.perf_counter()
            d1.copy_(h1, non_blocking=True)
            res = post(model(d1), sizes)[0]
            _ = [res["scores"].cpu(), res["labels"].cpu(), res["boxes"].cpu()]
            ts.append((time.perf_counter() - t0) * 1e3)
        lat_e2e = statistics.median(ts[10:])
    except Exception as ex:  # noqa
        lat_e2e = None

    # ---- per-kernel timing (CUDA events on the launch stream) for the roofline of the dominant kernel
    roof, table, prof = None, None, None
    if rank == 0:
        eng.forward(xs[0], want_aux=False)
        torch.cuda.synchronize()
        prof = eng.profile_ops(iters=5)
        pk = peaks()
        tot = sum(p[3] for p in prof)
        groups = {}
        for lab, fl, by, ms in prof:
            key = lab.split(".")[-1] if lab.startswith("block") or lab.startswith("dec") or lab.startswith("level") else lab
            if lab.startswith("block") and "." not in lab:
                key = "fc2"
            g = groups.setdefault(key, [0.0, 0.0, 0.0, 0])
            g[0] += ms; g[1] += fl; g[2] += by; g[3] += 1
        top = max(groups.items(), key=lambda kv: kv[1][0])
        name, (gms, gfl, gby, n) = top
        tens_t = gfl / (pk["bf16_tflops"] * 1e12) if gfl else 0.0
        hbm_t = gby / (pk["hbm_gbs"] * 1e9)
        if tens_t >= hbm_t:
            ach = gfl / (gms * 1e-3) / 1e12
            roof = {"kernel": name, "launches_per_step": n, "bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                    "frac": ach / pk["bf16_tflops"], "traffic": None, "share_of_step": gms / tot, "peak_source": pk["source"] + " (burst)"}
        else:
            ach = gby / (gms * 1e-3) / 1e9
            roof = {"kernel": name, "launches_per_step": n, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / pk["hbm_gbs"], "traffic": None, "share_of_step": gms / tot, "peak_source": pk["source"]}
        # DRAM traffic per launch of this kernel from a committed ncu --set full capture (profiles/kernel_traffic.json);
        # null when no capture exists for this config / batch / dtype.  Compare with the algorithmic bytes per launch.
        roof["algorithmic_bytes_per_launch"] = gby / n
        try:
            with open(os.path.join(ROOT, "profiles", "kernel_traffic.json")) as f:
                roof["traffic"] = json.load(f).get("%s:%d:%s:%s" % (cfg_name, batch, dtype_name, name))
        except Exception:
            pass
        if name.endswith("attn"):
            # attention at head dim 16/32 is bound by exp (MUFU, 16 ex2/clk/SM), not by the tensor pipe: report that too
            dh = (cfg.vit_dim // cfg.vit_heads) if name in ("glb_attn", "win_attn") else (cfg.hidden_dim // cfg.sa_nheads)
            gexp = gfl / (4.0 * dh) / (gms * 1e-3) / 1e9
            mufu_peak = 16 * 148 * 1.965                      # Gexp/s at the maximum SM clock
            roof["exp_bound"] = {"achieved_gexp_s": gexp, "peak_gexp_s": mufu_peak, "frac": gexp / mufu_peak,
                                 "note": "softmax exp count / MUFU.EX2 throughput (16/clk/SM x 148 SMs x 1.965 GHz)"}
        # per-op bandwidths come from back-to-back repeats of the same op (Engine::profile_ops): working sets below the
        # 126 MB L2 are L2-warm there, so "gbps" of a small op is NOT an HBM figure - it is labelled as such
        table = [{"op": k, "launches": v[3], "ms": v[0], "share": v[0] / tot, "gflop": v[1] / 1e9, "mbytes": v[2] / 1e6,
                  "tflops": (v[1] / (v[0] * 1e-3) / 1e12) if v[0] > 0 else 0, "gbps": (v[2] / (v[0] * 1e-3) / 1e9) if v[0] > 0 else 0,
                  "gbps_is_l2_warm": bool(v[2] / max(1, v[3]) < 126e6)}
                 for k, v in sorted(groups.items(), key=lambda kv: -kv[1][0])]
        if profile_out:
            with open(profile_out, "w") as f:
                json.dump({"config": cfg_name, "batch": batch, "dtype": dtype_name, "sum_ms": tot, "ops": table,
                           "per_op": [{"op": l, "ms": m, "gflop": fl / 1e9, "mbytes": by / 1e6} for l, fl, by, m in prof]}, f, indent=1)

    step_bytes = sum(p[2] for p in prof) if prof else 0.0
    tensor_frac = value * FLOPS_PER_IMAGE[cfg_name] / (peaks()["bf16_tflops_sustained"] * 1e12)
    config_extra = {"l2": "no flush needed: inputs alternate between two fp32 batches of %.0f MB and one step streams %.1f GB of "
                          "activations and weights through the kernels (>> 126 MB L2), so nothing survives from step to step"
                          % (in_bytes / 1e6, step_bytes / 1e9),
                    "cuda_graph": graph, "pdl": pdl, "weight_broadcast_bytes": bcast_bytes, "replicas_bit_identical": replicas_agree,
                    "model_gflop_per_image": FLOPS_PER_IMAGE[cfg_name] / 1e9, "whole_model_tensor_frac_of_sustained": tensor_frac}
    n_kernels = len(eng.ops())
    res = {"value": value, "ms_per_step": ms_total / steps, "e2e": e2e, "p50_latency_bs1_ms": lat, "p50_latency_bs1_e2e_postprocess_ms": lat_e2e,
           "roofline": roof, "top_ops": table[:8] if table else None, "n_kernels": n_kernels, "config_extra": config_extra,
           "whole_model_tensor_frac_of_sustained": tensor_frac,
           "clocks": sampler.summary(load_t0 + 0.05, load_t1) if (rank == 0 and clocks) else None}
    model._engine = None
    eng.close()
    del model, eng, xs
    torch.cuda.empty_cache()
    return res


if __name__ == "__main__":
    main()
