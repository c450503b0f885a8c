"""CPU tests of the frames entry point (lwdetr_forward_frames): a numpy restatement of the resize kernel's arithmetic
(csrc/resize.cu), with the coefficients computed in the kernel's order, is bit-identical to what the reference's callers
run on the host - torchvision's Resize([R, R]) on a PIL image - and the C ABI declares what the ctypes binding uses."""
import ctypes
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp
from PIL import Image
from torchvision import transforms

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PB = 22   # fixed-point bits of the taps


def coeffs(n_in, n_out):
    """Taps of one pass as a sparse [n_out, n_in] int64 matrix, every double operation in the kernel's order."""
    scale = n_in / n_out
    fs = max(scale, 1.0)
    support, ss = fs, 1.0 / fs
    rows, cols, vals = [], [], []
    for xx in range(n_out):
        c = (xx + 0.5) * scale
        xmin = max(int(c - support + 0.5), 0)
        n = min(int(c + support + 0.5), n_in) - xmin
        w = [max(0.0, 1.0 - abs((x + xmin - c + 0.5) * ss)) for x in range(n)]
        ww = 0.0
        for v in w:
            ww += v
        for x in range(n):
            v = w[x] / ww if ww != 0.0 else w[x]
            rows.append(xx)
            cols.append(xmin + x)
            vals.append(int(0.5 + v * (1 << PB)) if v >= 0 else int(-0.5 + v * (1 << PB)))
    return sp.csr_matrix((np.array(vals, np.int64), (rows, cols)), shape=(n_out, n_in))


def _pass(K, a):
    """One pass over the leading axis of a [n_in, ...] uint8 array -> [n_out, ...] uint8."""
    flat = a.reshape(a.shape[0], -1).astype(np.int64)
    out = (K @ flat + (1 << (PB - 1))) >> PB
    return np.clip(out, 0, 255).astype(np.uint8).reshape((K.shape[0],) + a.shape[1:])


def resize(img, R):
    """img uint8 [H, W, 3] -> [R, R, 3]: horizontal pass then vertical, except that very tall images (H > 100 W, shrinking
    in height) go vertical first, as Image.resize does."""
    H, W, _ = img.shape
    horizontal = (lambda x: _pass(coeffs(W, R), x.transpose(1, 0, 2)).transpose(1, 0, 2)) if W != R else (lambda x: x)
    vertical = (lambda x: _pass(coeffs(H, R), x)) if H != R else (lambda x: x)
    if H > 100 * W and R < H:
        return np.ascontiguousarray(horizontal(vertical(img)))
    return np.ascontiguousarray(vertical(horizontal(img)))


def sources(H, W, seed):
    """Seeded noise, a gradient with hard edges, all 0 and all 255."""
    rng = np.random.default_rng(seed)
    noise = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    y = np.arange(H)[:, None] * 255 // max(H - 1, 1)
    x = np.arange(W)[None, :] * 255 // max(W - 1, 1)
    grad = np.stack([y + 0 * x, x + 0 * y, (y + x) // 2], -1).astype(np.uint8)
    grad[(np.arange(H)[:, None] // 7 + np.arange(W)[None, :] // 11) % 5 == 0] = (255, 0, 255)   # hard edges
    return {"noise": noise, "gradient": grad, "zeros": np.zeros((H, W, 3), np.uint8), "full": np.full((H, W, 3), 255, np.uint8)}


SIDES = [448, 640, 896]


def source_sizes(R):
    return [(720, 1280), (1080, 1920), (2160, 3840), (4320, 7680), (240, 320), (1, 1), (640, 640),
            (R, 1000), (1000, R), (17, 2000), (8192, 8)]


@pytest.mark.parametrize("R", SIDES)
@pytest.mark.parametrize("k", range(11))
def test_restatement_matches_torchvision_resize_on_pil(R, k):
    H, W = source_sizes(R)[k]
    tf = transforms.Resize([R, R])
    for name, img in sources(H, W, seed=H * 31 + W).items():
        want = np.asarray(tf(Image.fromarray(img)))
        got = resize(img, R)
        assert got.shape == want.shape == (R, R, 3)
        bad = np.argwhere(got != want)
        assert bad.size == 0, "%dx%d -> %d, %s: %d values differ, first at (y, x, c) = %s" % (H, W, R, name, len(bad), tuple(bad[0]))


def test_identity_and_constant_frames_fall_out_of_the_formula():
    K = coeffs(640, 640).toarray()
    assert (K[:, :].max(1) == 1 << PB).all() and (K.sum(1) == 1 << PB).all()
    for n_in, n_out in ((1080, 640), (1, 896), (8192, 448), (240, 640)):
        s = coeffs(n_in, n_out).sum(1)
        assert (np.abs(s - (1 << PB)) <= 20).all()    # rounded taps: the sum stays within a few units of 2^22


# ------------------------------------------------------------------------------------------------ C ABI
def _header():
    with open(os.path.join(ROOT, "include", "lwdetr_b200.h")) as f:
        return f.read()


_CTYPES = {"const uint8_t*": ctypes.c_void_p, "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64}


def test_header_declares_frame_and_forward_frames():
    hdr = _header()
    m = re.search(r"LWDETR_API\s+int\s+lwdetr_forward_frames\s*\(([^;]*)\);", hdr)
    assert m, "lwdetr_forward_frames is not declared"
    args = [" ".join(a.split()) for a in m.group(1).split(",")]
    assert args[:4] == ["lwdetr_handle* h", "const lwdetr_frame* frames", "int B", "int img_size"]
    assert args[4:6] == ["const float mean[3]", "const float std[3]"]
    assert args[-1] == "void* stream" and len(args) == 11
    assert "#define LWDETR_MAX_FRAMES 1024" in hdr and "#define LWDETR_MAX_FRAME_SIDE 8192" in hdr


def test_ctypes_frame_matches_header_layout():
    from b200 import capi
    body = re.search(r"typedef struct \{([^}]*)\} lwdetr_frame;", _header()).group(1)
    fields = []
    for line in body.split(";")[:-1]:
        decl = re.sub(r"/\*.*?\*/", "", line, flags=re.S).strip()
        typ, names = re.match(r"((?:const\s+)?\w+\*?)\s+(.*)", decl).groups()
        fields += [(n.strip(), _CTYPES[typ]) for n in names.split(",")]
    header_struct = type("HeaderFrame", (ctypes.Structure,), {"_fields_": fields})
    assert [n for n, _ in fields] == [n for n, _ in capi.FrameDesc._fields_]
    for n, _ in fields:
        assert getattr(header_struct, n).offset == getattr(capi.FrameDesc, n).offset, n
    assert ctypes.sizeof(header_struct) == ctypes.sizeof(capi.FrameDesc) == 24
    assert (capi.MAX_FRAMES, capi.MAX_FRAME_SIDE) == (1024, 8192)


def test_library_exports_forward_frames():
    from b200 import capi
    assert "lwdetr_forward_frames" in capi.exported_symbols()
    assert hasattr(capi.lib(), "lwdetr_forward_frames")
    assert capi.lib().lwdetr_abi_version() == 1
