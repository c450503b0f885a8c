"""uint8 frames of any size through lwdetr_forward_frames on the device: the fused Pillow-exact resize + patch gather
against forward_at on frames resized by Pillow on the host, mixed batches, the whole forward, the drop-in recipe of
demo.py and the rejections of bad descriptors."""
import ctypes

import numpy as np
import pytest
import torch
from PIL import Image
from torchvision import transforms

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
SIDES = [448, 640, 896]


def source_sizes(R):
    return [(720, 1280), (1080, 1920), (2160, 3840), (4320, 7680), (240, 320), (1, 1), (640, 640),
            (R, 1000), (1000, R), (17, 2000), (8192, 8)]


def frames_np(H, W, seed):
    """Seeded noise, a gradient with hard edges, all 0 and all 255 (one batch)."""
    rng = np.random.default_rng(seed)
    noise = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    y = np.arange(H)[:, None] * 255 // max(H - 1, 1)
    x = np.arange(W)[None, :] * 255 // max(W - 1, 1)
    grad = np.stack([y + 0 * x, x + 0 * y, (y + x) // 2], -1).astype(np.uint8)
    grad[(np.arange(H)[:, None] // 7 + np.arange(W)[None, :] // 11) % 5 == 0] = (255, 0, 255)
    return [noise, grad, np.zeros((H, W, 3), np.uint8), np.full((H, W, 3), 255, np.uint8)]


def pil_resize(img, R):
    return np.asarray(transforms.Resize([R, R])(Image.fromarray(img)))


_ENGINES = {}


def tiny_engine(dt):
    from b200 import capi
    from b200.config import CONFIGS
    from b200.synth import synth_state_dict
    if dt not in _ENGINES:
        eng = capi.Engine(CONFIGS["tiny"], dt)
        eng.load_state_dict(synth_state_dict(CONFIGS["tiny"], 1))
        _ENGINES[dt] = eng
    return _ENGINES[dt]


def patch_matrix(eng, run, B, R):
    eng.clear_captures()
    cap = eng.capture("patch_gather", B * (R // 16) ** 2 * 768)
    out = run()
    torch.cuda.synchronize()
    got = eng.capture_results()["patch_gather"]
    eng.clear_captures()
    assert got is not None and got.numel() == cap.numel()
    return got.reshape(B * (R // 16) ** 2, 768).clone(), out


def first_mismatch(a, b, R):
    """(image, y, x, channel) of the first differing element of two window-major patch matrices."""
    r, k = (a != b).nonzero()[0].tolist()
    G = R // 16
    wh = G // 4
    img, rem = divmod(r, G * G)
    win, t = divmod(rem, wh * wh)
    Y, X = (win >> 2) * wh + t // wh, (win & 3) * wh + t % wh
    c, py, px = k // 256, (k % 256) // 16, k % 16
    return img, Y * 16 + py, X * 16 + px, c


def assert_same_patches(a, b, R, what):
    if not torch.equal(a, b):
        n = int((a != b).sum())
        raise AssertionError("%s: %d patch values differ, first at (image, y, x, channel) = %s" % (what, n, first_mismatch(a, b, R)))


# ------------------------------------------------------------------------------------------------ 1. patch matrix
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("R", SIDES)
@pytest.mark.parametrize("k", range(11))
def test_patch_matrix_equals_forward_at_on_pillow_resized(dt, R, k):
    H, W = source_sizes(R)[k]
    eng = tiny_engine(dt)
    srcs = frames_np(H, W, seed=H * 31 + W)
    frames = [torch.from_numpy(f).cuda() for f in srcs]
    resized = torch.from_numpy(np.stack([pil_resize(f, R) for f in srcs])).cuda()
    B = len(srcs)
    got, _ = patch_matrix(eng, lambda: eng.forward_frames(frames, img_size=R, want_aux=False), B, R)
    want, _ = patch_matrix(eng, lambda: eng.forward(resized, want_aux=False), B, R)
    assert_same_patches(got, want, R, "%dx%d -> %d" % (H, W, R))
    ops = {lab: by for lab, _, by in eng.ops()}
    # forward_at ran last: the op reports a [B,3,R,R] input again
    assert ops["patch_gather"] == 1.0 * B * 3 * R * R * 4 + 2.0 * B * (R // 16) ** 2 * 768


# ------------------------------------------------------------------------------------------------ 2. mixed batch
def test_mixed_batch_with_cropped_and_unaligned_frames_equals_single_calls():
    R = 640
    eng = tiny_engine(torch.float16)
    rng = np.random.default_rng(5)
    full = torch.from_numpy(rng.integers(0, 256, (900, 1700, 3), dtype=np.uint8)).cuda()
    crop = full[100:820, 37:1317]                              # 720 x 1280 view, row stride 5100 > 3 * 1280
    assert crop.stride(0) > 3 * crop.shape[1]
    raw = torch.from_numpy(rng.integers(0, 256, 1 + 333 * 517 * 3, dtype=np.uint8)).cuda()
    odd = raw[1:].view(333, 517, 3)                            # data pointer off 16-byte alignment
    assert odd.data_ptr() % 16 != 0
    frames = [crop, odd, torch.from_numpy(rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8)).cuda(),
              torch.from_numpy(rng.integers(0, 256, (240, 320, 3), dtype=np.uint8)).cuda(),
              torch.from_numpy(rng.integers(0, 256, (2160, 3840, 3), dtype=np.uint8)).cuda()]
    got, out = patch_matrix(eng, lambda: eng.forward_frames(frames, img_size=R), 5, R)
    out = {k: out[k].clone() for k in ("pred_logits", "pred_boxes")}
    T = (R // 16) ** 2
    for i, f in enumerate(frames):
        one, single = patch_matrix(eng, lambda: eng.forward_frames([f], img_size=R), 1, R)
        assert_same_patches(got[i * T:(i + 1) * T], one, R, "frame %d" % i)
        pil = torch.from_numpy(pil_resize(f.cpu().numpy(), R)).cuda()[None]
        at, _ = patch_matrix(eng, lambda: eng.forward(pil, want_aux=False), 1, R)
        assert_same_patches(one, at, R, "frame %d vs Pillow" % i)
        # one image's predictions do not depend on the rest of the batch beyond fp accumulation order
        assert (single["pred_boxes"][0] - out["pred_boxes"][i]).abs().max().item() < 2e-3
        assert (single["pred_logits"][0] - out["pred_logits"][i]).abs().max().item() < 5e-2


def test_batch_above_64_frames_takes_the_large_descriptor_list():
    """65 frames of 65 sizes: more descriptors than the small kernel-parameter list holds."""
    R = 448
    eng = tiny_engine(torch.float16)
    rng = np.random.default_rng(9)
    srcs = [rng.integers(0, 256, (17 + 13 * i, 900 - 11 * i, 3), dtype=np.uint8) for i in range(65)]
    frames = [torch.from_numpy(f).cuda() for f in srcs]
    resized = torch.from_numpy(np.stack([pil_resize(f, R) for f in srcs])).cuda()
    got, _ = patch_matrix(eng, lambda: eng.forward_frames(frames, img_size=R, want_aux=False), 65, R)
    want, _ = patch_matrix(eng, lambda: eng.forward(resized, want_aux=False), 65, R)
    assert_same_patches(got, want, R, "65 mixed frames")


# ------------------------------------------------------------------------------------------------ 3. end to end
def _all(out):
    t = {"pred_logits": out["pred_logits"], "pred_boxes": out["pred_boxes"], "enc_logits": out["enc_outputs"]["pred_logits"],
         "enc_boxes": out["enc_outputs"]["pred_boxes"], "topk": out["topk_index"]}
    for i, a in enumerate(out["aux_outputs"]):
        t["aux%d_logits" % i], t["aux%d_boxes" % i] = a["pred_logits"], a["pred_boxes"]
    return {k: v.clone() for k, v in t.items()}


def _assert_equal(a, b, what):
    for k in a:
        assert torch.equal(a[k], b[k]), "%s: %s differs" % (what, k)


@pytest.mark.parametrize("graph", [0, 1])
def test_small_b32_1080p_end_to_end_bit_identical(graph):
    from b200 import capi
    from b200.config import CONFIGS
    from b200.synth import synth_state_dict
    R, B = 640, 32
    eng = capi.Engine(CONFIGS["small"], torch.float16)
    eng.load_state_dict(synth_state_dict(CONFIGS["small"], 3))
    if graph:
        eng.set_option("cuda_graph", 1)
    rng = np.random.default_rng(11)
    batches = {}
    for H, W in ((1080, 1920), (720, 1280)):
        src = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(B)]
        batches[H] = (torch.from_numpy(np.stack(src)).cuda(), torch.from_numpy(np.stack([pil_resize(s, R) for s in src])).cuda())
    for H in (1080, 720, 1080):          # frames of a new size replay the same plan (and graph); forward_at interleaves
        frames, resized = batches[H]
        want = _all(eng.forward(resized))
        got = _all(eng.forward_frames(frames))
        again = _all(eng.forward_frames(frames))
        _assert_equal(got, want, "%dp graph=%d" % (H, graph))
        _assert_equal(again, want, "%dp repeated, graph=%d" % (H, graph))
    ops = {lab: by for lab, _, by in eng.ops()}
    assert ops["patch_gather"] == 3.0 * B * 1080 * 1920 + 2.0 * B * 40 * 40 * 768
    eng.close()


# ------------------------------------------------------------------------------------------------ 4. drop-in
def test_dropin_forward_frames_then_postprocess_equals_demo_recipe():
    from b200.config import CONFIGS
    from b200.synth import synth_state_dict
    from models.lwdetr import LWDETR, PostProcess
    from util.misc import nested_tensor_from_tensor_list
    cfg = CONFIGS["tiny"]
    model = LWDETR(cfg, compute_dtype=torch.float16).eval()
    model.load_state_dict(synth_state_dict(cfg, 2), strict=True)
    model.cuda()
    post = PostProcess(num_select=cfg.num_queries)
    H, W = 1080, 1920
    frame = np.random.default_rng(3).integers(0, 256, (H, W, 3), dtype=np.uint8)
    # demo.py:146-159: PIL -> Resize([640, 640]) -> ToTensor -> Normalize -> nested tensor -> model -> postprocessor
    tf = transforms.Compose([transforms.Resize([640, 640]), transforms.ToTensor(),
                             transforms.Normalize([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])])
    x = tf(Image.fromarray(frame))
    want = post(model(nested_tensor_from_tensor_list([x.cuda()])), torch.tensor([[H, W]], device="cuda"))[0]
    got = post(model.forward_frames([torch.from_numpy(frame)]), torch.tensor([[H, W]], device="cuda"))[0]
    for k in ("scores", "labels", "boxes"):
        assert torch.equal(got[k], want[k]), k
    # export mode: the tuple, at the configured size only
    model.export()
    assert isinstance(model.forward_frames(torch.from_numpy(frame)[None].cuda()), tuple)
    with pytest.raises(RuntimeError, match="export"):
        model.forward_frames([torch.from_numpy(frame)], img_size=512)


# ------------------------------------------------------------------------------------------------ 5. rejections
def _raw_call(eng, descs, R=640):
    from b200 import capi
    B = len(descs)
    arr = (capi.FrameDesc * B)(*descs)
    m, s = (ctypes.c_float * 3)(*capi.IMAGENET_MEAN), (ctypes.c_float * 3)(*capi.IMAGENET_STD)
    logits = torch.empty(B, 100, 91, device="cuda")
    boxes = torch.empty(B, 100, 4, device="cuda")
    rc = capi.lib().lwdetr_forward_frames(eng._h, ctypes.cast(arr, ctypes.c_void_p), B, R, ctypes.cast(m, ctypes.c_void_p),
                                          ctypes.cast(s, ctypes.c_void_p), capi.ptr(logits), capi.ptr(boxes), None, None,
                                          capi.stream_ptr())
    torch.cuda.synchronize()
    return rc, capi.lib().lwdetr_last_error().decode()


def test_rejections_leave_the_handle_usable():
    from b200 import capi
    eng = tiny_engine(torch.float16)
    buf = torch.zeros(64 * 64 * 3 + 64, dtype=torch.uint8, device="cuda")

    def desc(data, h, w, stride):
        return capi.FrameDesc(data, h, w, stride)

    good = desc(buf.data_ptr(), 64, 64, 192)
    want = eng.forward_frames([buf[:64 * 64 * 3].view(64, 64, 3)])["pred_logits"].clone()
    cases = [([desc(None, 64, 64, 192)], 640, "null data"),
             ([desc(buf.data_ptr(), 0, 64, 192)], 640, "sides must be in"),
             ([desc(buf.data_ptr(), 8193, 1, 3)], 640, "sides must be in"),
             ([desc(buf.data_ptr(), 64, 64, 191)], 640, "row_stride 191"),
             ([good], 700, "img_size 700"),
             ([good] * 1025, 640, "outside \\[1, 1024\\]")]
    for descs, R, msg in cases:
        rc, err = _raw_call(eng, descs, R)
        assert rc != 0 and re_search(msg, err), (msg, err)
        rc, err = _raw_call(eng, [good])
        assert rc == 0, err
    py_cases = [[torch.zeros(64, 64, 3, dtype=torch.float32, device="cuda")],       # not uint8
                [torch.zeros(3, 64, 64, dtype=torch.uint8, device="cuda")],         # CHW
                torch.zeros(2, 3, 64, 64, dtype=torch.uint8, device="cuda"),        # NCHW
                [torch.zeros(64, 64, 3, dtype=torch.uint8, device="cuda")[:, ::2]], # pixel stride 6
                [torch.zeros(64, 64, 3, dtype=torch.uint8)],                        # host tensor at the engine level
                [torch.zeros(1, 1, 3, dtype=torch.uint8, device="cuda")] * 1025]
    for frames in py_cases:
        with pytest.raises(RuntimeError):
            eng.forward_frames(frames)
    got = eng.forward_frames([buf[:64 * 64 * 3].view(64, 64, 3)])["pred_logits"]
    assert torch.equal(got, want)


def re_search(pattern, text):
    import re
    return re.search(pattern, text) is not None
