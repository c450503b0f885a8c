"""Parity ladder: CUDA engine (fp16 / bf16) vs the CPU oracle (fp32) on identical synthetic weights/inputs.

Prints / returns per-stage errors (SURVEY.md 8c tiers T1 pre-top-k tensors, T2 forced indices,
T3 free-running).  Runs on the GPU box:  python tools/parity_report.py small --batch 2 --dtype fp16
"""
import argparse
import dataclasses
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "lw-detr_b200"))

from b200 import capi  # noqa: E402
from b200.config import CONFIGS  # noqa: E402
from b200.synth import synth_images, synth_state_dict  # noqa: E402
from oracle import lwdetr_oracle as orc  # noqa: E402


def rel_l2(a, b):
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def ladder(name, batch, dtype, wseed=1, iseed=0, eng=None, img_size=640):
    """img_size: square input side; the engine keeps the configuration's own img_size and runs at img_size through
    lwdetr_forward_at, the oracle takes the level shapes and proposals of a config with img_size replaced."""
    cfg = CONFIGS[name]
    sd = synth_state_dict(cfg, wseed)
    x = synth_images(batch, iseed, img_size)
    own = eng is None
    if own:
        eng = capi.Engine(cfg, dtype)
        eng.load_state_dict(sd)
    cfg = dataclasses.replace(cfg, img_size=img_size)
    inter = {}
    ref = orc.forward(sd, cfg, x, inter=inter)
    xg = x.cuda()
    BT, C, d, S, nq = batch * cfg.tokens, cfg.vit_dim, cfg.hidden_dim, cfg.memory_len, cfg.num_queries
    caps = {"patch_embed": BT * C}
    for i in range(cfg.vit_depth):
        caps["block%d" % i] = BT * C
    for l in range(cfg.n_levels):
        caps["level%d" % l] = batch * S * d
    caps["enc_score"] = batch * S
    caps["query_pos"] = batch * nq * d
    for i in range(cfg.dec_layers):
        caps["dec%d" % i] = batch * nq * d
    eng.clear_captures()
    for k, n in caps.items():
        eng.capture(k, n)
    out_forced = eng.forward(xg, topk_override=inter["topk"])
    torch.cuda.synchronize()
    got = eng.capture_results()
    eng.clear_captures()
    rep = {"config": name, "batch": batch, "img_size": img_size, "dtype": str(dtype).replace("torch.", "")}
    t1 = {}
    t1["patch_embed"] = rel_l2(got["patch_embed"].reshape(BT, C), inter["patch"].reshape(BT, C))
    for i in range(cfg.vit_depth):
        t1["block%d" % i] = rel_l2(got["block%d" % i].reshape(BT, C), inter["block%d" % i].reshape(BT, C))
    mem = got["level%d" % (cfg.n_levels - 1)].reshape(batch, S, d)
    t1["memory"] = rel_l2(mem, inter["memory"])
    start = 0
    for l, (h, w) in enumerate(cfg.level_shapes):
        t1["level%d" % l] = rel_l2(mem[:, start:start + h * w], inter["level%d" % l])
        start += h * w
    t1["enc_score_maxabs"] = (got["enc_score"].reshape(batch, S) - inter["enc_score"]).abs().max().item()
    rep["T1"] = t1
    t2 = {"query_pos": rel_l2(got["query_pos"].reshape(batch, nq, d), inter["query_pos"])}
    for i in range(cfg.dec_layers):
        t2["dec%d" % i] = rel_l2(got["dec%d" % i].reshape(batch, nq, d), inter["dec%d" % i])

    def cmp(o, r, pre=""):
        return {pre + "logits_rel_l2": rel_l2(o["pred_logits"].cpu(), r["pred_logits"]),
                pre + "logits_maxabs": (o["pred_logits"].cpu() - r["pred_logits"]).abs().max().item(),
                pre + "boxes_maxabs": (o["pred_boxes"].cpu() - r["pred_boxes"]).abs().max().item()}

    t2.update(cmp(out_forced, ref))
    t2.update(cmp(out_forced["enc_outputs"], ref["enc_outputs"], "enc_"))
    for i, (a, b) in enumerate(zip(out_forced["aux_outputs"], ref["aux_outputs"])):
        t2.update(cmp(a, b, "aux%d_" % i))
    t2["topk_echo_ok"] = bool((out_forced["topk_index"].cpu().long() == inter["topk"]).all())
    rep["T2"] = t2
    # T3 free running
    out_free = eng.forward(xg)
    torch.cuda.synchronize()
    ti = out_free["topk_index"].cpu().long()
    set_agree, slot_same = [], []
    for b in range(batch):
        a, r = set(ti[b].tolist()), set(inter["topk"][b].tolist())
        set_agree.append(len(a & r) / float(nq))
        slot_same.append((ti[b] == inter["topk"][b]).float().mean().item())
    same = (ti == inter["topk"])
    t3 = {"set_agreement_min": min(set_agree), "slot_agreement_mean": sum(slot_same) / batch}
    if same.any():
        t3["slot_aligned_enc_boxes_maxabs"] = (out_free["enc_outputs"]["pred_boxes"].cpu() - ref["enc_outputs"]["pred_boxes"])[same].abs().max().item()
        t3["slot_aligned_enc_logits_maxabs"] = (out_free["enc_outputs"]["pred_logits"].cpu() - ref["enc_outputs"]["pred_logits"])[same].abs().max().item()
    t3["finite"] = bool(torch.isfinite(out_free["pred_logits"]).all() and torch.isfinite(out_free["pred_boxes"]).all())
    rep["T3"] = t3
    if own:
        eng.close()
    return rep


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=["tiny"])
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--dtype", default="fp16,bf16")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.set_num_threads(os.cpu_count())
    reps = []
    for name in a.configs:
        for dt in a.dtype.split(","):
            try:
                rep = ladder(name, a.batch, {"fp16": torch.float16, "bf16": torch.bfloat16}[dt])
            except Exception as e:  # keep going: the report is a diagnostic
                rep = {"config": name, "dtype": dt, "error": repr(e)}
            reps.append(rep)
            print(json.dumps(rep, indent=1), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(reps, f, indent=1)


def baseline_parity(name, batch, dtype, chunk=4, wseed=1, iseed=11):
    """Oracle comparison of EVERY image of a BASELINE.json batch (configs[1..4]) through the C ABI: the oracle runs in
    chunks of `chunk` images (it is batch-independent per image), the engine runs the whole batch at once - i.e. with
    the GEMM tilings, attention grids and persistent-CTA splits bench.py measures.  T2: two-stage indices forced to the
    oracle's, outputs compared element-wise; T3: free-running selected-set agreement per image."""
    cfg = CONFIGS[name]
    sd = synth_state_dict(cfg, wseed)
    x = synth_images(batch, iseed)
    refs, topks, mems, scores = [], [], [], []
    for lo in range(0, batch, chunk):
        inter = {}
        r = orc.forward(sd, cfg, x[lo:lo + chunk], inter=inter)
        refs.append(r)
        topks.append(inter["topk"])
        mems.append(inter["memory"])
        scores.append(inter["enc_score"])
    topk = torch.cat(topks)
    cat = lambda key: torch.cat([r[key] for r in refs])
    ref = {"pred_logits": cat("pred_logits"), "pred_boxes": cat("pred_boxes"),
           "enc_logits": torch.cat([r["enc_outputs"]["pred_logits"] for r in refs]),
           "enc_boxes": torch.cat([r["enc_outputs"]["pred_boxes"] for r in refs]),
           "aux_logits": [torch.cat([r["aux_outputs"][i]["pred_logits"] for r in refs]) for i in range(cfg.dec_layers - 1)],
           "aux_boxes": [torch.cat([r["aux_outputs"][i]["pred_boxes"] for r in refs]) for i in range(cfg.dec_layers - 1)]}
    eng = capi.Engine(cfg, dtype)
    eng.load_state_dict(sd)
    xg = x.cuda()
    S, d, nq = cfg.memory_len, cfg.hidden_dim, cfg.num_queries
    eng.capture("level%d" % (cfg.n_levels - 1), batch * S * d)
    eng.capture("enc_score", batch * S)
    forced = eng.forward(xg, topk_override=topk)
    torch.cuda.synchronize()
    got = eng.capture_results()
    eng.clear_captures()
    mem = got["level%d" % (cfg.n_levels - 1)].reshape(batch, S, d)
    memref = torch.cat(mems)
    per_img = lambda a, b: ((a - b).flatten(1).norm(dim=1) / (b.flatten(1).norm(dim=1) + 1e-12))
    rep = {"config": name, "batch": batch, "dtype": str(dtype).replace("torch.", "")}
    rep["memory_rel_l2_max"] = per_img(mem, memref).max().item()
    rep["enc_score_maxabs"] = (got["enc_score"].reshape(batch, S) - torch.cat(scores)).abs().max().item()
    rep["topk_echo_ok"] = bool((forced["topk_index"].cpu().long() == topk).all())
    fl, fb = forced["pred_logits"].cpu(), forced["pred_boxes"].cpu()
    rep["logits_rel_l2_max"] = per_img(fl, ref["pred_logits"]).max().item()       # worst image
    rep["logits_rel_l2"] = rel_l2(fl, ref["pred_logits"])
    rep["logits_maxabs"] = (fl - ref["pred_logits"]).abs().max().item()
    rep["boxes_maxabs"] = (fb - ref["pred_boxes"]).abs().max().item()
    rep["enc_logits_maxabs"] = (forced["enc_outputs"]["pred_logits"].cpu() - ref["enc_logits"]).abs().max().item()
    rep["enc_boxes_maxabs"] = (forced["enc_outputs"]["pred_boxes"].cpu() - ref["enc_boxes"]).abs().max().item()
    rep["aux_logits_maxabs"] = max((forced["aux_outputs"][i]["pred_logits"].cpu() - ref["aux_logits"][i]).abs().max().item() for i in range(cfg.dec_layers - 1))
    rep["aux_boxes_maxabs"] = max((forced["aux_outputs"][i]["pred_boxes"].cpu() - ref["aux_boxes"][i]).abs().max().item() for i in range(cfg.dec_layers - 1))
    free = eng.forward(xg)
    torch.cuda.synchronize()
    ti = free["topk_index"].cpu().long()
    rep["set_agreement_min"] = min(len(set(ti[b].tolist()) & set(topk[b].tolist())) / float(nq) for b in range(batch))
    rep["finite"] = bool(torch.isfinite(free["pred_logits"]).all() and torch.isfinite(free["pred_boxes"]).all())
    same = (ti == topk)
    if same.any():
        rep["slot_aligned_enc_boxes_maxabs"] = (free["enc_outputs"]["pred_boxes"].cpu() - ref["enc_boxes"])[same].abs().max().item()
        rep["slot_aligned_enc_logits_maxabs"] = (free["enc_outputs"]["pred_logits"].cpu() - ref["enc_logits"])[same].abs().max().item()
    eng.close()
    return rep
