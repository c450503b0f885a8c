"""Inference at square input sides other than 640 on the device: the parity ladder against the oracle, the engine against
the reference's own outputs (tests/golden/ref_res.npz), the kernels at the shapes 640 never reaches, and the public
module switching resolutions under one engine."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tools"))
sys.path.insert(0, HERE)

from test_model_gpu import TOL  # noqa: E402

DTYPES = [torch.float16, torch.bfloat16]
# (config, R, batch) of tests/golden/ref_res.npz
RES_CASES = [("tiny", 448, 2), ("small", 512, 1), ("medium", 576, 1), ("large", 768, 1), ("xlarge", 896, 1)]


def _rel_l2(a, b):
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _gold():
    return np.load(os.path.join(HERE, "golden", "ref_res.npz"))


# ------------------------------------------------------------------------------------------------ model parity
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("name,R,batch", RES_CASES)
def test_parity_ladder_at_other_resolutions(name, R, batch, dt):
    """The bars of test_model_gpu.test_parity_ladder, unchanged, at the sizes the reference trains at."""
    import parity_report
    rep = parity_report.ladder(name, batch, dt, img_size=R)
    tol = TOL[dt]
    t1, t2, t3 = rep["T1"], rep["T2"], rep["T3"]
    for k, v in t1.items():
        if k.startswith("block") or k == "patch_embed":
            assert v <= tol["block"], (k, v)
        elif k.startswith("level") or k == "memory":
            assert v <= tol["memory"], (k, v)
    assert t1["enc_score_maxabs"] <= tol["score"], t1
    assert t2["topk_echo_ok"]
    for k, v in t2.items():
        if k.endswith("logits_rel_l2"):
            assert v <= tol["logits_rel"], (k, v)
        elif k.endswith("logits_maxabs"):
            assert v <= tol["logits_abs"], (k, v)
        elif k.endswith("boxes_maxabs"):
            assert v <= tol["boxes"], (k, v)
        elif k.startswith("dec") or k == "query_pos":
            assert v <= tol["dec"], (k, v)
    assert t3["finite"]
    assert t3["set_agreement_min"] >= 0.95, t3
    if "slot_aligned_enc_boxes_maxabs" in t3:
        assert t3["slot_aligned_enc_boxes_maxabs"] <= 2 * tol["boxes"], t3
        assert t3["slot_aligned_enc_logits_maxabs"] <= 2 * tol["logits_abs"], t3


def _sample(t, n):
    """The strided sample tools/make_goldens.py stores (sample()): every (numel // n)-th element, n of them."""
    f = t.detach().reshape(-1).float().cpu()
    return f[::max(1, f.numel() // n)][:n]


def _check_against_golden(out, g, case, tol):
    gl, gb = torch.from_numpy(g[case + "_pred_logits"]), torch.from_numpy(g[case + "_pred_boxes"])
    logits = _sample(out["pred_logits"], len(gl))      # the fixture keeps a strided sample of the logits
    assert _rel_l2(logits, gl) <= tol["logits_rel"]
    assert (logits - gl).abs().max().item() <= tol["logits_abs"]
    assert (out["pred_boxes"].cpu() - gb).abs().max().item() <= tol["boxes"]
    assert (out["enc_outputs"]["pred_boxes"].cpu() - torch.from_numpy(g[case + "_enc_boxes"])).abs().max().item() <= tol["boxes"]


@pytest.mark.parametrize("dt", DTYPES)
def test_engine_matches_reference_golden_at_448(dt):
    """tiny at 448 x 448 (28 x 28 tokens, 49-token windows) through lwdetr_forward_at against the reference's own output,
    with the two-stage selection forced to the oracle's (SURVEY.md 8c tier T2)."""
    import dataclasses
    from b200 import capi
    from b200.config import CONFIGS
    from b200.synth import synth_images, synth_state_dict
    from oracle import lwdetr_oracle as orc
    g = _gold()
    B, wseed, iseed, R = (int(v) for v in g["tiny448_meta"])
    cfg = CONFIGS["tiny"]
    sd = synth_state_dict(cfg, wseed)
    x = synth_images(B, iseed, R)
    inter = {}
    orc.forward(sd, dataclasses.replace(cfg, img_size=R), x, inter=inter)
    eng = capi.Engine(cfg, dt)
    eng.load_state_dict(sd)
    forced = eng.forward(x.cuda(), topk_override=inter["topk"])
    _check_against_golden(forced, g, "tiny448", TOL[dt])
    free = eng.forward(x.cuda())
    for b in range(B):
        assert len(set(free["topk_index"][b].tolist()) & set(inter["topk"][b].tolist())) >= 0.95 * cfg.num_queries
    eng.close()


@pytest.mark.parametrize("dt", DTYPES)
def test_padded_batch_at_512_matches_reference_golden(dt):
    """A 512 x 512 and a 448 x 384 image: the module runs the batch at its 512 extent with the padding mask, as the
    reference does (tests/golden/ref_res.npz 'pad512')."""
    import dataclasses
    from b200 import capi
    from b200.config import CONFIGS
    from b200.synth import synth_images, synth_state_dict
    from models.lwdetr import LWDETR
    from oracle import lwdetr_oracle as orc
    g = _gold()
    B, wseed, iseed, extent = (int(v) for v in g["pad512_meta"])
    cfg = CONFIGS["tiny"]
    x = synth_images(B, iseed, extent).clone()
    mask = torch.zeros(B, extent, extent, dtype=torch.bool)
    for b, (h, w) in enumerate(g["pad512_valid"]):
        mask[b, int(h):, :] = True
        mask[b, :, int(w):] = True
        x[b][:, mask[b]] = 0
    sd = synth_state_dict(cfg, wseed)
    inter = {}
    orc.forward(sd, dataclasses.replace(cfg, img_size=extent), x, inter=inter, mask=mask)
    eng = capi.Engine(cfg, dt)
    eng.load_state_dict(sd)
    forced = eng.forward(x.cuda(), mask=mask.cuda(), topk_override=inter["topk"])
    _check_against_golden(forced, g, "pad512", TOL[dt])
    free = eng.forward(x.cuda(), mask=mask.cuda())
    free = {k: free[k].clone() for k in ("pred_logits", "pred_boxes", "topk_index")}
    for b in range(B):
        assert len(set(free["topk_index"][b].tolist()) & set(inter["topk"][b].tolist())) >= 0.95 * cfg.num_queries
    model = LWDETR(cfg, compute_dtype=dt).eval()
    model.load_state_dict(sd, strict=True)
    model.cuda()
    imgs = [x[b][:, : int(h), : int(w)].cuda() for b, (h, w) in enumerate(g["pad512_valid"])]
    out = model(imgs)
    assert torch.equal(out["pred_logits"], free["pred_logits"]) and torch.equal(out["pred_boxes"], free["pred_boxes"])
    eng.close()


# ------------------------------------------------------------------------------------------------ kernels at the new shapes
def _tol(dt):
    return 3e-3 if dt == torch.float16 else 2e-2


REL_L2 = {torch.float16: 1e-3, torch.bfloat16: 8e-3}


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("dh", [16, 32, 64])
@pytest.mark.parametrize("nseq,seqlen", [(32, 49), (32, 121), (32, 144), (32, 196),     # windows (16 per image, B = 2) at 448, 704, 768, 896
                                         (2, 784), (1, 3136)])                           # global attention at 448 and 896
def test_attention_at_other_resolutions(dt, dh, nseq, seqlen):
    """Windows of 144-196 tokens take two query tiles in the slot kernel (dh 16 / 32) and leave attn_short_kernel's
    112-token range at dh 64; global attention spans 784-3136 tokens."""
    from b200 import capi
    heads = 12
    g = torch.Generator(device="cuda").manual_seed(seqlen * 7 + dh)
    C = heads * dh
    qkv = (torch.randn(nseq * seqlen, 3 * C, device="cuda", generator=g) * 1.5).to(dt)
    out = torch.full((nseq * seqlen, C), float("nan"), device="cuda", dtype=dt)
    scale = dh ** -0.5
    capi.attention(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], out, nseq, seqlen, heads, dh, scale)
    q, k, v = [t.float().reshape(nseq, seqlen, heads, dh).transpose(1, 2) for t in (qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:])]
    ref = ((q * scale) @ k.transpose(-2, -1)).softmax(-1) @ v
    ref = ref.transpose(1, 2).reshape(nseq * seqlen, C)
    assert torch.isfinite(out.float()).all()
    assert (out.float() - ref).abs().max().item() <= _tol(dt) * ref.abs().max().item()
    assert _rel_l2(out.float(), ref) <= REL_L2[dt]
    row_err = (out.float() - ref).norm(dim=1) / (ref.norm(dim=1) + 1e-6)
    assert row_err.max().item() <= 8 * REL_L2[dt], row_err.max().item()


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("shapes", [[(96, 96), (24, 24)], [(112, 112), (28, 28)]])     # large / xlarge levels at 768 and 896
def test_msda_forward_p3_levels_above_8192_tokens(dt, shapes):
    """P3 levels of 9216 and 12544 tokens: corner tokens need the 14-bit field of the packed sample word, and 112-wide
    rows cut the level into 8 bands plus one for P5."""
    from b200 import capi
    from oracle import lwdetr_oracle as orc
    B, Lq, M, L, P = 2, 300, 24, 2, 4
    g = torch.Generator().manual_seed(shapes[0][0])
    d = M * 16
    S = sum(h * w for h, w in shapes)
    value = torch.randn(B, S, d, generator=g).to(dt)
    ol = torch.cat([torch.randn(B * Lq, M * L * P * 2, generator=g) * 2.0, torch.randn(B * Lq, M * L * P, generator=g) * 2.0], 1).to(dt)
    ref_box = torch.rand(B * Lq, 4, generator=g) * torch.tensor([1.2, 1.2, 0.6, 0.6]) - torch.tensor([0.1, 0.1, 0.0, 0.0])
    out = torch.full((B * Lq, d), float("nan"), dtype=dt, device="cuda")
    capi.msda_forward(capi.value_to_head_major(value.cuda().reshape(B * S, d), B, S, M), ol.cuda(), ref_box.cuda(), out,
                      B, S, Lq, M, L, P, shapes)
    off = ol[:, :M * L * P * 2].float().reshape(B, Lq, M, L, P, 2)
    aw = ol[:, M * L * P * 2:].float().reshape(B, Lq, M, L * P).softmax(-1).reshape(B, Lq, M, L, P)
    rb = ref_box.reshape(B, Lq, 4)
    loc = rb[:, :, None, None, None, :2] + off / P * rb[:, :, None, None, None, 2:] * 0.5
    ref = orc.msda_core(value.float().reshape(B, S, M, 16), shapes, loc, aw).reshape(B * Lq, d)
    assert (out.float().cpu() - ref).abs().max().item() <= _tol(dt) * max(ref.abs().max().item(), 1.0)
    assert _rel_l2(out.float().cpu(), ref) <= REL_L2[dt]


def test_msda_forward_rejects_levels_above_16384_tokens():
    from b200 import capi
    B, Lq, M, L, P, shapes = 1, 4, 1, 1, 2, [(129, 128)]
    S = 129 * 128
    v = torch.zeros(B, M, S, 16, device="cuda", dtype=torch.float16)
    ol = torch.zeros(B * Lq, 3 * M * L * P, device="cuda", dtype=torch.float16)
    out = torch.empty(B * Lq, M * 16, device="cuda", dtype=torch.float16)
    with pytest.raises(RuntimeError, match="16384"):
        capi.msda_forward(v, ol, torch.zeros(B * Lq, 4, device="cuda"), out, B, S, Lq, M, L, P, shapes)


def test_topk_at_13328_tokens():
    """xlarge at 896: S = 112^2 + 28^2 memory tokens."""
    from b200 import capi
    B, S, k = 2, 13328, 300
    g = torch.Generator(device="cuda").manual_seed(S)
    score = torch.randn(B, S, device="cuda", generator=g)
    score[1, 7] = score[1, 13000] = score[1].max() + 1.0     # a tie at the top, far apart: the lower index comes first
    idx = capi.topk(score, k).long()
    vals, ref = torch.sort(score, dim=1, descending=True, stable=True)
    assert torch.equal(torch.gather(score, 1, idx), vals[:, :k])
    assert torch.equal(idx, ref[:, :k])
    assert idx[1, 0].item() == 7 and idx[1, 1].item() == 13000


# ------------------------------------------------------------------------------------------------ one module, many sizes
def _pred(out):
    return {k: out[k].clone() for k in ("pred_logits", "pred_boxes")}


def _equal(a, b):
    return torch.equal(a["pred_logits"], b["pred_logits"]) and torch.equal(a["pred_boxes"], b["pred_boxes"])


def _tiny_module(seed=1):
    from b200.config import CONFIGS
    from b200.synth import synth_state_dict
    from models.lwdetr import LWDETR
    model = LWDETR(CONFIGS["tiny"], compute_dtype=torch.float16).eval()
    model.load_state_dict(synth_state_dict(CONFIGS["tiny"], seed), strict=True)
    return model.cuda()


@pytest.mark.parametrize("graph", [0, 1])
def test_module_switches_resolution_under_one_engine(graph):
    """640 -> 512 -> 896 -> 640 through one module (one handle, one weight arena): each change re-plans, and both 640
    results are bit-identical to a fresh module's, eager and with CUDA graphs."""
    from b200.synth import synth_images
    xs = {R: synth_images(2, R, R).cuda() for R in (640, 512, 896)}
    fresh = _tiny_module()
    want640 = _pred(fresh(xs[640]))
    model = _tiny_module()
    eng = model.engine()
    if graph:
        eng.set_option("cuda_graph", 1)
    got = []
    for R in (640, 512, 896, 640):
        out = _pred(model(xs[R]))
        if graph:      # the first forward of a plan runs eagerly; the second replays the graph
            again = _pred(model(xs[R]))
            assert _equal(again, out), R
        assert out["pred_logits"].shape == (2, 100, 91) and torch.isfinite(out["pred_logits"]).all()
        got.append(out)
    assert _equal(got[0], want640) and _equal(got[3], want640)
    assert not torch.equal(got[1]["pred_logits"], got[2]["pred_logits"])
    # a fresh engine that has only ever seen 512 / 896 gives the same results as the one that switched
    for i, R in ((1, 512), (2, 896)):
        assert _equal(_pred(_tiny_module()(xs[R])), got[i]), R


def test_module_uint8_and_rejected_sizes_at_other_resolutions():
    from b200 import capi
    model = _tiny_module()
    g = torch.Generator().manual_seed(2)
    u8 = torch.randint(0, 256, (2, 512, 512, 3), generator=g, dtype=torch.uint8)
    mean, std = torch.tensor(capi.IMAGENET_MEAN), torch.tensor(capi.IMAGENET_STD)
    f32 = ((u8.float() / 255.0 - mean) / std).permute(0, 3, 1, 2).contiguous()
    a = _pred(model(f32.cuda()))
    b = _pred(model(u8.cuda()))
    assert _equal(a, b)
    for bad in (torch.zeros(1, 3, 960, 960), torch.zeros(1, 3, 700, 700), torch.zeros(2, 3, 512, 512, dtype=torch.uint8),
                torch.zeros(1, 384, 384, 3, dtype=torch.uint8)):
        with pytest.raises(RuntimeError):
            model(bad.cuda())
    # the C ABI rejects a side outside the supported set on its own
    eng = model.engine()
    desc = capi.InputDesc()
    x = torch.zeros(1, 3, 960, 960, device="cuda")
    desc.images, desc.format = x.data_ptr(), capi.IN_F32_NCHW
    logits = torch.empty(1, 100, 91, device="cuda")
    boxes = torch.empty(1, 100, 4, device="cuda")
    rc = capi.lib().lwdetr_forward_at(eng._h, ctypes.byref(desc), 960, 1, capi.ptr(logits), capi.ptr(boxes), None, None, capi.stream_ptr())
    assert rc != 0 and b"img_size 960" in capi.lib().lwdetr_last_error()
    # export mode keeps the reference's fixed 40 x 40 position table (vit.py:328-332)
    model.export()
    with pytest.raises(RuntimeError, match="export"):
        model(f32.cuda())
    assert isinstance(model(torch.zeros(1, 3, 640, 640).cuda()), tuple)


def test_reload_after_other_resolution_rebuilds_position_table():
    """Weights loaded after a forward at 512 give what a fresh engine with those weights gives at 512."""
    from b200 import capi
    from b200.config import CONFIGS
    from b200.synth import synth_images, synth_state_dict
    cfg = CONFIGS["tiny"]
    x = synth_images(2, 3, 512).cuda()
    eng = capi.Engine(cfg, torch.float16)
    eng.load_state_dict(synth_state_dict(cfg, 1))
    first = _pred(eng.forward(x))
    eng.load_state_dict(synth_state_dict(cfg, 2))
    reloaded = _pred(eng.forward(x))
    ref = capi.Engine(cfg, torch.float16)
    ref.load_state_dict(synth_state_dict(cfg, 2))
    want = _pred(ref.forward(x))
    assert _equal(reloaded, want) and not torch.equal(first["pred_logits"], reloaded["pred_logits"])
    eng.close()
    ref.close()


# ------------------------------------------------------------------------------------------------ two ranks
def _nccl_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from b200 import capi
        from b200.config import CONFIGS
        from b200.dist import broadcast_engine_weights
        from b200.synth import synth_images, synth_state_dict
        cfg = CONFIGS["tiny"]
        x = synth_images(2, 4, 512).cuda()
        eng = capi.Engine(cfg, torch.float16)
        eng.load_state_dict(synth_state_dict(cfg, 1 if rank == 0 else 7))    # rank 1: placeholder values, same layout
        if rank == 1:
            eng.forward(x)                                                       # plans 512 (position table from seed 7)
            torch.cuda.synchronize()
        broadcast_engine_weights(eng, torch.device("cuda", rank), src=0)
        out = eng.forward(x)
        q.put((rank, out["pred_logits"].cpu(), out["pred_boxes"].cpu()))
        eng.close()
    finally:
        dist.destroy_process_group()


def test_broadcast_after_planning_other_resolution_two_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = sorted((q.get(timeout=600) for _ in range(2)), key=lambda r: r[0])
    finally:
        for p in procs:
            p.join(timeout=120)
            if p.is_alive():
                p.terminate()
                p.join()
    assert torch.equal(res[0][1], res[1][1]) and torch.equal(res[0][2], res[1][2])
