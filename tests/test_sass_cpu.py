"""The shipped library really takes the Blackwell path: SASS mnemonic counts per kernel (cuobjdump, no GPU needed).
UTCHMMA = tcgen05.mma, UTMALDG = TMA tensor load, UBLKCP = cp.async.bulk, LDTM / STTM = tcgen05.ld / st, HMMA = legacy mma.sync."""
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "lw-detr_b200", "lib", "liblwdetr_b200.so")


@pytest.fixture(scope="module")
def table():
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    if not os.path.exists(LIB):
        sys.path.insert(0, ROOT)
        import __graft_entry__
        __graft_entry__.build()
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sass_proof.py"), LIB], capture_output=True, text=True, check=True).stdout
    rows, cols = {}, None
    for line in out.splitlines():
        if line.startswith("#"):
            continue
        if line.startswith("kernel"):
            cols = line.split()[1:]
            continue
        m = re.match(r"(.*?)\s+((?:\d+\s*)+)$", line)
        if m and cols:
            vals = [int(v) for v in m.group(2).split()]
            if len(vals) == len(cols):
                rows[m.group(1).strip()] = dict(zip(cols, vals))
    assert rows, out[:500]
    return rows


def _sel(table, prefix):
    return {k: v for k, v in table.items() if prefix in k}


def test_attention_slot_kernels_are_exactly_the_dispatched_set_and_tcgen05_tma_only(table):
    ks = _sel(table, "attn_slots_kernel<")
    # {fp16, bf16} x {head dim 16, 32} x {one tile per sequence, longer sequences}: nothing else is compiled
    assert set(ks) == {"sl::attn_slots_kernel<%s, %d, %s>" % (t, dh, lg)
                       for t in ("__half", "__nv_bfloat16") for dh in (16, 32) for lg in ("false", "true")}, sorted(ks)
    for name, c in ks.items():
        assert c["UTCHMMA"] > 0 and c["UTMALDG"] > 0 and c["LDTM"] > 0 and c["STTM"] > 0, name
        assert c["HMMA"] == 0 and c["LDGSTS"] == 0, name


def test_attention_tc_kernels_are_head_dim_64_tcgen05_tma_only(table):
    ks = _sel(table, "attn_tc_kernel<")
    assert set(ks) == {"attn_tc_kernel<__half, 64>", "attn_tc_kernel<__nv_bfloat16, 64>"}, sorted(ks)
    for name, c in ks.items():
        assert c["UTCHMMA"] > 0 and c["UTMALDG"] > 0 and c["LDTM"] > 0, name
        assert c["HMMA"] == 0, name


def test_gemm_family_is_tcgen05_tma(table):
    ks = _sel(table, "gemm_tc_kernel<")
    assert len(ks) >= 24
    for name, c in ks.items():
        assert c["UTCHMMA"] > 0 and c["UTMALDG"] > 0 and c["LDTM"] > 0, name
        assert c["HMMA"] == 0, name


def test_deformable_gather_streams_with_bulk_copies(table):
    ks = _sel(table, "msda_fwd_kernel<")
    assert ks
    for name, c in ks.items():
        assert c["UBLKCP"] > 0 and c["FFMA2"] > 0, name


def test_legacy_mma_sync_only_where_documented(table):
    """mma.sync (HMMA) is allowed only in attn.cu's kernels: decoder self-attention, head-dim-64 windows, unpacked q/k/v."""
    for name, c in table.items():
        if c["HMMA"] > 0:
            assert name.startswith("attn_kernel<") or name.startswith("attn_short_kernel<"), name
