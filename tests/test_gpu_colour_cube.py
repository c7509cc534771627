"""GPU tests: every output kernel's colour step on all 2^24 (Y, Cb, Cr) triples, and every kernel's DC-only blocks on
each (c0, q0) of the sweep, byte for byte against the expectations of tests/colour_cube.py (pinned to the oracle by
tests/test_colour_cube.py).

Tier A (one 4096 x 4096 file per sampling, each holding every triple once) runs through the packed colour step
hjd_color_n in the CUDA-core and tensor-core fused kernels, in its BGR form for BMP output, and in the unfused
hjd_k_color (KEEP_PLANES); tier B (8192 x 8192 4:2:0 at 1/2) through the scaled kernel's sc_ycc; tier C (DC-only
sweeps) through every kernel's DC-only path.  Each batch asserts the idct_variant bits, so that no test passes through
a kernel other than the one it names."""
import numpy as np
import pytest

from tests import colour_cube as cc

pytestmark = pytest.mark.gpu

A_FLAGS = ("default", "tensor_core", "cuda_core", "keep_planes", "bmp", "bmp_tensor_core", "gray")
C_FLAGS = ("keep_planes", "tensor_core", "cuda_core", "gray", "scale_1_2", "scale_1_4", "scale_1_8",
           "gray_scale_1_2", "gray_scale_1_4", "gray_scale_1_8")


def _flags(hjd, name):
    f = {"default": 0, "tensor_core": hjd.FLAG_TENSOR_CORE_IDCT, "cuda_core": hjd.FLAG_CUDA_CORE_IDCT,
         "keep_planes": hjd.FLAG_KEEP_PLANES, "bmp": hjd.FLAG_BMP_OUT,
         "bmp_tensor_core": hjd.FLAG_BMP_OUT | hjd.FLAG_TENSOR_CORE_IDCT, "gray": hjd.FLAG_GRAY_OUT}
    if name in f:
        return f[name]
    gray = name.startswith("gray_")
    scale = {"2": hjd.FLAG_SCALE_1_2, "4": hjd.FLAG_SCALE_1_4, "8": hjd.FLAG_SCALE_1_8}[name[-1]]
    return scale | (hjd.FLAG_GRAY_OUT if gray else 0)


def _variants(name):
    """The idct_variant values (include/hjd.h) the flag set allows: bit 0 tensor-core fused kernel, bit 1 CUDA-core
    fused kernel, bit 2 scaled kernel, bit 3 luma-only kernel; 0 for KEEP_PLANES (the unfused kernels).  Without a
    kernel flag the batch's chunks may take either fused kernel."""
    if name.startswith("gray_scale") or name.startswith("scale"):
        return {4 | (8 if name.startswith("gray") else 0)}
    return {"default": {1, 2, 3}, "tensor_core": {1}, "cuda_core": {2}, "keep_planes": {0}, "bmp": {1, 2, 3},
            "bmp_tensor_core": {1}, "gray": {8}}[name]


def _bmp_to_rgb(bmp, w, h):
    pad = (4 - (w * 3) % 4) % 4
    rows = np.frombuffer(bmp, dtype=np.uint8, offset=54).reshape(h, w * 3 + pad)[::-1, :w * 3]
    return rows.reshape(h, w, 3)[:, :, ::-1]


def _report(case, got, want, what):
    """None when equal, else the number of wrong samples and wrong (Y, Cb, Cr) triples and the first few as
    (Y, Cb, Cr, channel, got, want)."""
    if got.shape != want.shape:
        return f"{case.name} {what}: shape {got.shape}, want {want.shape}"
    bad = got != want
    if not bad.any():
        return None
    if got.ndim == 3:
        yy, xx, ch = np.nonzero(bad)
        tri = (case.yc[yy, xx].astype(np.int64) << 16) | (case.cbc[yy, xx].astype(np.int64) << 8) | case.crc[yy, xx]
        first = [(int(case.yc[y, x]), int(case.cbc[y, x]), int(case.crc[y, x]), "RGB"[c], int(got[y, x, c]),
                  int(want[y, x, c])) for y, x, c in zip(yy[:8], xx[:8], ch[:8])]
        return (f"{case.name} {what}: {int(bad.sum())} samples wrong, {np.unique(tri).size} distinct triples; "
                f"first (Y, Cb, Cr, channel, got, want): {first}")
    yy, xx = np.nonzero(bad)
    first = [(int(y), int(x), int(got[y, x]), int(want[y, x])) for y, x in zip(yy[:8], xx[:8])]
    return f"{case.name} {what}: {int(bad.sum())} samples wrong; first (row, column, got, want): {first}"


def _run(hjd, cases, name):
    """Decode the cases' files in one batch under the flag set and compare everything it outputs."""
    flags = _flags(hjd, name)
    errors = []
    with hjd.BatchDecoder(0, flags) as d:
        d.upload([c.jpg for c in cases])
        d.decode()
        st = d.status()
        assert (st == 0).all(), (name, st)
        assert d.idct_variant in _variants(name), (name, d.idct_variant)
        slab = d.plane_slab() if flags & hjd.FLAG_KEEP_PLANES else None
        for i, c in enumerate(cases):
            if flags & hjd.FLAG_GRAY_OUT:
                errors.append(_report(c, d.gray(i), c.yc, "gray"))
            elif flags & hjd.FLAG_BMP_OUT:
                h, w = c.yc.shape
                errors.append(_report(c, _bmp_to_rgb(d.bmp(i), w, h), c.rgb(), "bmp"))
            else:
                errors.append(_report(c, d.rgb(i), c.rgb(), "rgb"))
            if slab is not None:
                for k, (got, want) in enumerate(zip(d.planes(i, slab), (c.y, c.cb, c.cr))):
                    if want is not None:
                        errors.append(_report(c, got, want, ("Y", "Cb", "Cr")[k]))
    errors = [e for e in errors if e]
    assert not errors, "\n".join(errors)


@pytest.fixture(scope="module")
def tier_a():
    return [cc.tier_a(s) for s in ("444", "422", "440", "420", "gray")]


@pytest.mark.parametrize("flag_set", A_FLAGS)
def test_tier_a_every_triple(hjd, tier_a, flag_set):
    _run(hjd, tier_a, flag_set)


def test_tier_b_scaled_every_triple(hjd):
    _run(hjd, [cc.tier_b()], "scale_1_2")


@pytest.fixture(scope="module")
def tier_c():
    return cc.tier_c()


@pytest.mark.parametrize("flag_set", C_FLAGS)
def test_tier_c_dc_only_blocks(hjd, tier_c, flag_set):
    n = 8 >> {"2": 1, "4": 2, "8": 3}.get(flag_set[-1], 0)
    _run(hjd, [f.case(n) for f in tier_c], flag_set)
