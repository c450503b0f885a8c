"""Kernel-level GPU tests through the C ABI: attention, LayerNorm, deformable attention, top-k.
The checker is the CPU oracle's math (oracle/lwdetr_oracle.py) or plain fp32 torch of the same op."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DTYPES = [torch.float16, torch.bfloat16]


def _tol(dt):
    return 3e-3 if dt == torch.float16 else 2e-2


def _rel_l2(a, b):
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


# rel-L2 bounds next to the max-abs ones (a single wrong low-magnitude row passes a max-abs / max|ref| test):
# 16-bit rounding of P and of the output gives ~3e-4 (fp16) / ~2.5e-3 (bf16) on these shapes
REL_L2 = {torch.float16: 1e-3, torch.bfloat16: 8e-3}


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("nseq,seqlen,heads,dh", [(32, 100, 12, 16), (2, 1600, 12, 16), (16, 100, 12, 32), (1, 1600, 12, 32),
                                                  (16, 100, 12, 64), (1, 1600, 12, 64), (3, 300, 8, 32), (2, 100, 8, 32),
                                                  (2, 300, 12, 32), (5, 37, 4, 16),
                                                  # attn_tc.cu (packed qkv, seqlen >= 512, dh 64): ragged tails, single-tile last CTA;
                                                  # dh 32 at these lengths: slot kernel, ragged tails
                                                  (2, 700, 6, 32), (3, 640, 4, 64), (2, 520, 4, 32), (1, 1153, 4, 64),
                                                  # slot kernel (attn_slots.cu: packed qkv, dh 16 / 32, any length): ragged query and key
                                                  # tails, more (sequence, head, query tile) items than slots, single-item launches
                                                  (3, 300, 4, 16), (2, 129, 4, 16), (1, 1153, 4, 16), (2, 513, 12, 16), (1, 64, 4, 16), (7, 128, 4, 16),
                                                  (640, 100, 12, 16), (70, 100, 12, 32), (3, 1, 4, 16), (2, 65, 4, 32)])
def test_attention_matches_softmax_reference(dt, nseq, seqlen, heads, dh):
    from b200 import capi
    g = torch.Generator(device="cuda").manual_seed(seqlen + dh)
    C = heads * dh
    qkv = (torch.randn(nseq * seqlen, 3 * C, device="cuda", generator=g) * 1.5).to(dt)
    out = torch.full((nseq * seqlen, C), float("nan"), device="cuda", dtype=dt)
    scale = dh ** -0.5
    capi.attention(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], out, nseq, seqlen, heads, dh, scale)
    q, k, v = [t.float().reshape(nseq, seqlen, heads, dh).transpose(1, 2) for t in (qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:])]
    ref = ((q * scale) @ k.transpose(-2, -1)).softmax(-1) @ v
    ref = ref.transpose(1, 2).reshape(nseq * seqlen, C)
    err = (out.float() - ref).abs().max().item()
    assert err <= _tol(dt) * ref.abs().max().item(), err
    assert _rel_l2(out.float(), ref) <= REL_L2[dt]
    # per-row bound: no query row may be off by more than a few 16-bit ulps of its own magnitude (measured worst row 4.8e-3 fp16
    # at 1153 keys: the rounding of P, averaged over the keys, against a row norm that is itself an average)
    row_err = (out.float() - ref).norm(dim=1) / (ref.norm(dim=1) + 1e-6)
    assert row_err.max().item() <= 8 * REL_L2[dt], row_err.max().item()


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("dh", [16, 32, 64])
def test_attention_late_dominant_keys(dt, dh):
    """Keys whose scores dwarf everything seen before arrive late in the sequence: the lazily tracked row maximum of
    the tcgen05 kernel has to move (O rescaled in TMEM) several times, and rows must still normalise exactly."""
    from b200 import capi
    nseq, seqlen, heads = 2, 1600, 4
    g = torch.Generator(device="cuda").manual_seed(dh)
    C = heads * dh
    qkv = torch.randn(nseq * seqlen, 3 * C, device="cuda", generator=g)
    for start, gain in ((300, 4.0), (900, 10.0), (1500, 25.0)):
        for s0 in range(nseq):
            qkv[s0 * seqlen + start:s0 * seqlen + start + 7, C:2 * C] *= gain
    qkv = qkv.to(dt)
    out = torch.full((nseq * seqlen, C), float("nan"), device="cuda", dtype=dt)
    scale = dh ** -0.5
    capi.attention(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], out, nseq, seqlen, heads, dh, scale)
    q, k, v = [t.float().reshape(nseq, seqlen, heads, dh).transpose(1, 2) for t in (qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:])]
    ref = ((q * scale) @ k.transpose(-2, -1)).softmax(-1) @ v
    ref = ref.transpose(1, 2).reshape(nseq * seqlen, C)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    assert err <= _tol(dt) * ref.abs().max().item(), err
    assert _rel_l2(out.float(), ref) <= REL_L2[dt]


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("rows,C,eps", [(3200, 192, 1e-6), (1000, 256, 1e-5), (777, 384, 1e-6), (64, 768, 1e-6)])
def test_layernorm(dt, rows, C, eps):
    from b200 import capi
    g = torch.Generator(device="cuda").manual_seed(C)
    xb = (torch.randn(rows, C + 64, device="cuda", generator=g) * 2 + 0.5).to(dt)
    x = xb[:, :C]
    w = torch.randn(C, device="cuda", generator=g)
    b = torch.randn(C, device="cuda", generator=g)
    y = torch.empty(rows, C, device="cuda", dtype=dt)
    capi.layernorm(x, y, w, b, eps)
    ref = F.layer_norm(x.float(), (C,), w, b, eps)
    assert (y.float() - ref).abs().max().item() <= _tol(dt) * ref.abs().max().item()
    assert _rel_l2(y.float(), ref) <= (5e-4 if dt == torch.float16 else 4e-3)


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("B,Lq,M,L,P,shapes", [(1, 2, 2, 2, 2, [(6, 4), (3, 2)]),      # models/ops/test.py:27-34 shapes
                                               (3, 300, 16, 1, 2, [(40, 40)]),
                                               (2, 300, 24, 2, 4, [(80, 80), (20, 20)]),
                                               (2, 100, 16, 1, 4, [(40, 40)])])
def test_msda_forward_matches_oracle(dt, B, Lq, M, L, P, shapes):
    from b200 import capi
    from oracle import lwdetr_oracle as orc
    g = torch.Generator().manual_seed(3 + Lq)
    D, d = 16, M * 16
    S = sum(h * w for h, w in shapes)
    nlayers = 3
    value_all = torch.randn(B, S, nlayers * d, generator=g).to(dt)          # 3 layers side by side, use the middle one
    offs = torch.randn(B * Lq, M * L * P * 2, generator=g) * 2.0
    logit = torch.randn(B * Lq, M * L * P, generator=g) * 2.0
    ol = torch.cat([offs, logit], 1).to(dt)
    ref_box = torch.rand(B * Lq, 4, generator=g) * torch.tensor([1.2, 1.2, 0.6, 0.6]) - torch.tensor([0.1, 0.1, 0.0, 0.0])
    out = torch.full((B * Lq, d), float("nan"), dtype=dt, device="cuda")
    vg = value_all.cuda()
    # the engine's layout: all layers' values head-major in one buffer [B][layer][M][S][16]; use the middle layer's slice
    hm = vg.reshape(B, S, nlayers, M, 16).permute(0, 2, 3, 1, 4).contiguous()
    capi.msda_forward(hm[:, 1], ol.cuda(), ref_box.cuda(), out, B, S, Lq, M, L, P, shapes, v_image_stride=nlayers * M * S * 16)
    # oracle on the same rounded inputs (ops/modules/ms_deform_attn.py:118-131 + msda core)
    value = value_all[..., d:2 * d].float().reshape(B, S, M, D)
    off = ol[:, :M * L * P * 2].float().reshape(B, Lq, M, L, P, 2)
    aw = ol[:, M * L * P * 2:].float().reshape(B, Lq, M, L * P).softmax(-1).reshape(B, Lq, M, L, P)
    rb = ref_box.reshape(B, Lq, 4)
    loc = rb[:, :, None, None, None, :2] + off / P * rb[:, :, None, None, None, 2:] * 0.5
    ref = orc.msda_core(value, shapes, loc, aw).reshape(B * Lq, d)
    err = (out.float().cpu() - ref).abs().max().item()
    assert err <= _tol(dt) * max(ref.abs().max().item(), 1.0), err
    assert _rel_l2(out.float().cpu(), ref) <= (1e-3 if dt == torch.float16 else 8e-3)


@pytest.mark.parametrize("dt", DTYPES)
def test_msda_forward_valid_ratios(dt):
    """Padded batches scale the reference boxes per level by the valid ratios (transformer.py:352-353)."""
    from b200 import capi
    from oracle import lwdetr_oracle as orc
    B, Lq, M, L, P, shapes = 2, 300, 24, 2, 4, [(80, 80), (20, 20)]
    g = torch.Generator().manual_seed(11)
    d, S = M * 16, sum(h * w for h, w in shapes)
    value = torch.randn(B, S, d, generator=g).to(dt)
    ol = torch.cat([torch.randn(B * Lq, M * L * P * 2, generator=g) * 2.0, torch.randn(B * Lq, M * L * P, generator=g)], 1).to(dt)
    ref_box = torch.rand(B * Lq, 4, generator=g) * torch.tensor([1.0, 1.0, 0.5, 0.5])
    vr = torch.tensor([[[1.0, 1.0], [1.0, 1.0]], [[0.8, 0.65], [0.8, 0.7]]])
    out = torch.full((B * Lq, d), float("nan"), dtype=dt, device="cuda")
    capi.msda_forward(capi.value_to_head_major(value.cuda().reshape(B * S, d), B, S, M), ol.cuda(), ref_box.cuda(), out, B, S, Lq, M, L, P, shapes,
                      valid_ratio=vr.cuda().contiguous())
    off = ol[:, :M * L * P * 2].float().reshape(B, Lq, M, L, P, 2)
    aw = ol[:, M * L * P * 2:].float().reshape(B, Lq, M, L * P).softmax(-1).reshape(B, Lq, M, L, P)
    rb = ref_box.reshape(B, Lq, 1, 4) * torch.cat([vr, vr], -1)[:, None]                     # [B, Lq, L, 4]
    loc = rb[:, :, None, :, None, :2] + off / P * rb[:, :, None, :, None, 2:] * 0.5
    ref = orc.msda_core(value.float().reshape(B, S, M, 16), shapes, loc, aw).reshape(B * Lq, d)
    assert (out.float().cpu() - ref).abs().max().item() <= _tol(dt) * max(ref.abs().max().item(), 1.0)


def _op_inputs(N, S, M, D, Lq, L, P, dt, seed=3):
    """models/ops/test.py:37-41 recipe."""
    torch.manual_seed(seed)
    value = (torch.rand(N, S, M, D).cuda() * 0.01).to(dt)
    loc = torch.rand(N, Lq, M, L, P, 2).cuda().to(dt)
    aw = torch.rand(N, Lq, M, L, P).cuda() + 1e-5
    aw = (aw / aw.sum(-1, keepdim=True).sum(-2, keepdim=True)).to(dt)
    return value, loc, aw


@pytest.mark.parametrize("dt", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("N,M,D,Lq,L,P,shapes", [(1, 2, 2, 2, 2, 2, [(6, 4), (3, 2)]),             # models/ops/test.py:27-31
                                                 (2, 2, 30, 2, 2, 2, [(6, 4), (3, 2)]),            # channel counts of test.py:111
                                                 (2, 2, 32, 2, 2, 2, [(6, 4), (3, 2)]),
                                                 (1, 2, 71, 2, 2, 2, [(6, 4), (3, 2)]),
                                                 (2, 16, 16, 300, 1, 2, [(40, 40)]),               # small / medium decoder shapes
                                                 (2, 24, 16, 300, 2, 4, [(80, 80), (20, 20)]),      # large / xlarge
                                                 (2, 8, 32, 100, 4, 4, [(32, 32), (16, 16), (8, 8), (4, 4)])])   # Deformable-DETR default
def test_ms_deform_attn_forward_operator(dt, N, M, D, Lq, L, P, shapes):
    """The reference operator's interface (ms_deform_attn.h:19-35) replayed with models/ops/test.py's recipe against the
    reference's own checker ms_deform_attn_core_pytorch (= oracle msda_core, pinned to the grid_sample form on CPU)."""
    from b200 import capi
    from oracle import lwdetr_oracle as orc
    sh = torch.as_tensor(shapes, dtype=torch.long).cuda()
    lsi = torch.cat((sh.new_zeros((1,)), sh.prod(1).cumsum(0)[:-1]))
    S = int(sh.prod(1).sum())
    value, loc, aw = _op_inputs(N, S, M, D, Lq, L, P, dt)
    out = capi.ms_deform_attn_forward(value, sh, lsi, loc, aw, im2col_step=2 if N <= 2 else 64)
    assert out.shape == (N, Lq, M * D) and out.dtype == dt
    ref = orc.msda_core(value.double().cpu(), shapes, loc.double().cpu(), aw.double().cpu())
    if dt == torch.float32:
        assert torch.allclose(out.cpu().double(), ref, rtol=1e-2, atol=1e-3)         # the reference's own float criterion (test.py:82)
        assert (out.cpu().double() - ref).abs().max().item() <= 2e-8 + 1e-5 * ref.abs().max().item()
    else:
        assert (out.cpu().double() - ref).abs().max().item() <= _tol(dt) * ref.abs().max().item()


def test_ms_deform_attn_forward_error_behaviour():
    """Same failures as the reference op: CPU tensors, non-contiguous tensors, batch not divisible by im2col_step."""
    from b200 import capi
    sh = torch.as_tensor([(6, 4), (3, 2)], dtype=torch.long).cuda()
    lsi = torch.cat((sh.new_zeros((1,)), sh.prod(1).cumsum(0)[:-1]))
    value, loc, aw = _op_inputs(3, 30, 2, 16, 2, 2, 2, torch.float32)
    with pytest.raises(RuntimeError, match="CPU"):
        capi.ms_deform_attn_forward(value.cpu(), sh, lsi, loc, aw)
    with pytest.raises(RuntimeError, match="contiguous"):
        capi.ms_deform_attn_forward(value.transpose(1, 2), sh, lsi, loc, aw)
    with pytest.raises(RuntimeError, match="im2col_step"):
        capi.ms_deform_attn_forward(value, sh, lsi, loc, aw, im2col_step=2)        # 3 % 2 != 0  (ms_deform_attn_cuda.cu:50-52)
    out = capi.ms_deform_attn_forward(value, sh, lsi, loc, aw, im2col_step=64)     # min(B, step) = 3 divides 3
    assert torch.isfinite(out).all()


@pytest.mark.parametrize("B,S,k", [(2, 1600, 300), (3, 6800, 300), (1, 1600, 100), (2, 50, 50)])
def test_topk_sorted_indices(B, S, k):
    from b200 import capi
    g = torch.Generator(device="cuda").manual_seed(S)
    score = torch.randn(B, S, device="cuda", generator=g)
    score[0, 5] = score[0, 9]                       # a tie: lower index first
    idx = capi.topk(score, k).long()
    vals, ref = torch.sort(score, dim=1, descending=True, stable=True)
    assert torch.equal(torch.gather(score, 1, idx), vals[:, :k])
    assert torch.equal(idx, ref[:, :k])


def _torch_postprocess(logits, boxes, target_sizes, k):
    """lwdetr.py:515-544 in plain torch (fp32)."""
    ncls = logits.shape[2]
    scores, flat = torch.topk(logits.sigmoid().flatten(1), k, dim=1)
    query, labels = flat // ncls, flat % ncls
    cx, cy, w, h = boxes.unbind(-1)
    xyxy = torch.stack([cx - 0.5 * w, cy - 0.5 * h, cx + 0.5 * w, cy + 0.5 * h], dim=-1)
    xyxy = torch.gather(xyxy, 1, query.unsqueeze(-1).expand(-1, -1, 4))
    img_h, img_w = target_sizes.unbind(1)
    return scores, labels, xyxy * torch.stack([img_w, img_h, img_w, img_h], dim=1)[:, None, :]


@pytest.mark.parametrize("B,nq,ncls,k", [(3, 300, 91, 300), (2, 100, 91, 100), (1, 300, 91, 100), (2, 900, 20, 300)])
def test_postprocess_matches_reference_math(B, nq, ncls, k):
    from b200 import capi
    g = torch.Generator(device="cuda").manual_seed(nq + k)
    logits = torch.randn(B, nq, ncls, device="cuda", generator=g) * 3.0
    boxes = torch.rand(B, nq, 4, device="cuda", generator=g) * 0.5 + 0.1
    sizes = torch.tensor([[480.0, 640.0], [640.0, 427.0], [333.0, 500.0]], device="cuda")[:B]
    scores, labels, xyxy = capi.postprocess(logits, boxes, sizes, k)
    rs, rl, rb = _torch_postprocess(logits, boxes, sizes, k)
    assert torch.allclose(scores, rs, rtol=2e-6, atol=1e-7)
    assert (scores[:, 1:] <= scores[:, :-1]).all()
    same = labels.long() == rl
    # a different order is only legitimate between scores that round to (almost) the same fp32 sigmoid
    gap = torch.minimum((rs - torch.roll(rs, 1, 1)).abs(), (rs - torch.roll(rs, -1, 1)).abs())
    assert (same | (gap < 1e-6)).all()
    assert same.float().mean() > 0.99
    assert torch.allclose(xyxy[same], rb[same], rtol=1e-6, atol=1e-4)


def test_postprocess_ties_and_module_surface():
    """Heavily quantised logits: thousands of exact ties.  The selected score VALUES must still be torch's, every emitted
    (label, box) must belong to a (query, class) pair with exactly that score, and PostProcess returns the reference's types."""
    from b200 import capi
    from models.lwdetr import PostProcess
    g = torch.Generator(device="cuda").manual_seed(5)
    B, nq, ncls, k = 2, 300, 91, 300
    logits = (torch.randn(B, nq, ncls, device="cuda", generator=g) * 2).round() / 2
    boxes = torch.rand(B, nq, 4, device="cuda", generator=g) * 0.5 + 0.1
    sizes = torch.tensor([[480.0, 640.0], [600.0, 400.0]], device="cuda")
    scores, labels, xyxy = capi.postprocess(logits, boxes, sizes, k)
    rs = torch.topk(logits.sigmoid().flatten(1), k, dim=1)[0]
    assert torch.allclose(scores, rs, rtol=2e-6, atol=1e-7)
    sig = logits.sigmoid()
    scale = torch.stack([sizes[:, 1], sizes[:, 0], sizes[:, 1], sizes[:, 0]], 1)
    for b in range(B):
        cx, cy, w, h = boxes[b].unbind(-1)
        cand = torch.stack([cx - 0.5 * w, cy - 0.5 * h, cx + 0.5 * w, cy + 0.5 * h], -1) * scale[b]      # [nq, 4]
        d = (cand[None, :, :] - xyxy[b][:, None, :]).abs().amax(-1)                                       # [k, nq]
        q = d.argmin(1)
        assert (d.gather(1, q[:, None]) < 1e-3).all()
        assert torch.allclose(sig[b, q, labels[b].long()], scores[b], rtol=2e-6, atol=1e-7)
    # ties go to the lower flat index: the emitted (query, class) pairs of equal score are in increasing order
    res = PostProcess(num_select=k)({"pred_logits": logits, "pred_boxes": boxes}, sizes)
    assert len(res) == B and res[0]["labels"].dtype == torch.int64 and res[0]["boxes"].shape == (k, 4)
    assert torch.equal(res[1]["scores"], scores[1])


@pytest.mark.parametrize("name", ["tiny", "small", "large"])
def test_postprocess_matches_reference_golden(name):
    """The fused device PostProcess against the REFERENCE's PostProcess output on the reference's golden predictions."""
    import os
    import numpy as np
    from b200 import capi
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    g, p = np.load(os.path.join(gold, "ref_%s.npz" % name)), np.load(os.path.join(gold, "ref_postprocess.npz"))
    logits, boxes = torch.from_numpy(g["pred_logits"]).cuda(), torch.from_numpy(g["pred_boxes"]).cuda()
    k = int(p[name + "_num_select"][0])
    scores, labels, xyxy = capi.postprocess(logits, boxes, torch.from_numpy(p[name + "_sizes"]).cuda(), k)
    rs, rl, rb = [torch.from_numpy(p[name + s]).cuda() for s in ("_scores", "_labels", "_boxes")]
    assert torch.allclose(scores, rs, rtol=2e-6, atol=1e-7)
    same = labels.long() == rl
    gap = torch.minimum((rs - torch.roll(rs, 1, 1)).abs(), (rs - torch.roll(rs, -1, 1)).abs())
    assert (same | (gap < 1e-6)).all() and same.float().mean() > 0.98
    assert torch.allclose(xyxy[same], rb[same], rtol=1e-6, atol=1e-3)


def _autograd_reference(value, shapes, loc, aw, grad_out):
    """Gradients of the oracle's msda_core (pinned to the grid_sample form / the reference's ms_deform_attn_core_pytorch)
    by torch autograd in float64 on the CPU."""
    from oracle import lwdetr_oracle as orc
    v, l, a = [t.detach().double().cpu().requires_grad_(True) for t in (value, loc, aw)]
    out = orc.msda_core(v, shapes, l, a)
    out.backward(grad_out.double().cpu())
    return out.detach(), v.grad, l.grad, a.grad


@pytest.mark.parametrize("N,M,D,Lq,L,P,shapes", [(1, 2, 2, 2, 2, 2, [(6, 4), (3, 2)]),            # models/ops/test.py:27-31
                                                 (2, 2, 30, 2, 2, 2, [(6, 4), (3, 2)]),           # test.py:111 channel counts
                                                 (2, 2, 71, 2, 2, 2, [(6, 4), (3, 2)]),
                                                 (2, 16, 16, 100, 1, 2, [(40, 40)]),
                                                 (1, 24, 16, 50, 2, 4, [(80, 80), (20, 20)])])
def test_ms_deform_attn_backward_operator(N, M, D, Lq, L, P, shapes):
    """ms_deform_attn_backward (ms_deform_attn.h:37-60) against autograd through the checker the reference itself uses
    (test.py:85-108 compares against numerical gradients of the same function)."""
    from b200 import capi
    sh = torch.as_tensor(shapes, dtype=torch.long).cuda()
    lsi = torch.cat((sh.new_zeros((1,)), sh.prod(1).cumsum(0)[:-1]))
    S = int(sh.prod(1).sum())
    value, loc, aw = _op_inputs(N, S, M, D, Lq, L, P, torch.float32, seed=7)
    value = value * 100.0                                                # O(1) values: gradients well above fp32 noise
    loc = (loc * 1.2 - 0.1).contiguous()                                 # some samples fall outside the image
    g = torch.Generator(device="cuda").manual_seed(1)
    grad_out = torch.randn(N, Lq, M * D, device="cuda", generator=g)
    gv, gl, ga = capi.ms_deform_attn_backward(value, sh, lsi, loc, aw, grad_out, im2col_step=64)
    _, rv, rl, ra = _autograd_reference(value, shapes, loc, aw, grad_out)
    for got, ref, what in ((gv, rv, "grad_value"), (gl, rl, "grad_sampling_loc"), (ga, ra, "grad_attn_weight")):
        err = (got.double().cpu() - ref).abs().max().item()
        assert err <= 2e-5 * max(1.0, ref.abs().max().item()), (what, err)


def test_reference_msdeformattnfunction_binds_to_this_library():
    """models/ops/test.py replayed through the calls the reference's autograd Function makes
    (functions/ms_deform_attn_func.py:23-50: `import MultiScaleDeformableAttention as MSDA`, then
    MSDA.ms_deform_attn_forward / _backward with its argument order): they resolve to the drop-in module and run on the
    sm_100a kernels.  The forward is compared with what the reference's checker ms_deform_attn_core_pytorch returned on
    the same inputs (tests/golden/ref_msda_checker.npz, tools/make_goldens.py --live-only)."""
    import importlib
    import os
    import sys
    import numpy as np
    mod = sys.modules.get("MultiScaleDeformableAttention")
    if mod is None or not hasattr(mod, "ms_deform_attn_forward"):
        sys.modules.pop("MultiScaleDeformableAttention", None)
        mod = importlib.import_module("MultiScaleDeformableAttention")    # lw-detr_b200/MultiScaleDeformableAttention.py
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_msda_checker.npz"))
    N, M, D, Lq, L, P = 1, 2, 2, 2, 2, 2                                   # test.py:27-31
    shapes = torch.as_tensor([(6, 4), (3, 2)], dtype=torch.long).cuda()
    assert torch.equal(shapes.cpu(), torch.from_numpy(g["shapes"]))
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    S = sum([(H * W).item() for H, W in shapes])
    torch.manual_seed(3)
    for i, cast in enumerate((lambda t: t.double(), lambda t: t)):        # check_forward_equal_with_pytorch_double / _float
        value = torch.rand(N, S, M, D).cuda() * 0.01
        loc = torch.rand(N, Lq, M, L, P, 2).cuda()
        aw = torch.rand(N, Lq, M, L, P).cuda() + 1e-5
        aw /= aw.sum(-1, keepdim=True).sum(-2, keepdim=True)
        for t, k in ((value, "value"), (loc, "loc"), (aw, "aw")):        # the inputs the checker saw
            assert torch.equal(t.cpu(), torch.from_numpy(g["%s%d" % (k, i)])), k
        ref = torch.from_numpy(g["out%d" % i])
        out = mod.ms_deform_attn_forward(cast(value), shapes, lsi, cast(loc), cast(aw), 2).detach().cpu()
        assert out.dtype == ref.dtype
        assert torch.allclose(out, ref, rtol=1e-2, atol=1e-3)              # test.py:82
        assert (out - ref).abs().max().item() < 1e-7
    # gradients: the backward call the reference Function makes (test.py:85-108 uses gradcheck on the same call)
    value = torch.rand(N, S, M, 8).cuda()
    loc = torch.rand(N, Lq, M, L, P, 2).cuda()
    aw = (torch.rand(N, Lq, M, L, P).cuda() + 1e-5)
    aw = aw / aw.sum(-1, keepdim=True).sum(-2, keepdim=True)
    out = mod.ms_deform_attn_forward(value, shapes, lsi, loc, aw, 2)
    gout = torch.randn_like(out)
    gv, gl, ga = mod.ms_deform_attn_backward(value, shapes, lsi, loc, aw, gout.contiguous(), 2)
    _, rv, rl, ra = _autograd_reference(value, [(6, 4), (3, 2)], loc, aw, gout)
    assert (gv.double().cpu() - rv).abs().max().item() < 1e-5
    assert (gl.double().cpu() - rl).abs().max().item() < 1e-4
    assert (ga.double().cpu() - ra).abs().max().item() < 1e-5
