"""CPU tests of the colour-cube and DC-only expectations (tests/colour_cube.py) against the oracle.

The colour step's whole input space is 2^24 (Y, Cb, Cr) triples and a DC-only block's is the pair (c0, q0), so both
are pinned exhaustively here: the numpy restatements against the oracle's own functions on every input, the files of
tiers A and B to hold every triple exactly once, and each file's oracle decode to equal its constructed expectation.
tests/test_gpu_colour_cube.py then compares the GPU kernels with the same expectations byte for byte."""
import numpy as np
import pytest

from tests import colour_cube as cc
from tests import scaled_port as sp


@pytest.fixture(scope="module")
def cube():
    return sp.ycc_cube().reshape(-1, 3)


def test_ycc_to_rgb_is_the_oracles_on_the_whole_cube(cube):
    y, cb, cr = cc.cube_triples()
    assert np.array_equal(cc.ycc_to_rgb(y, cb, cr), cube)


def _wrong(got, cube, channel=None):
    bad = got != (cube if channel is None else cube[:, channel])
    return int(bad.any(axis=1).sum()) if bad.ndim == 2 else int(bad.sum())


def test_cube_separates_the_alternative_formulations(cube):
    """Each formulation below differs from the reference on a few out-of-gamut triples only, and the golden fixtures
    hold none of them.  The counts pin that the cube keeps reaching those triples."""
    f32 = np.float32
    y, cb, cr = cc.cube_triples()
    yi, cbi, cri = y.astype(np.int64), cb.astype(np.int32) - 128, cr.astype(np.int32) - 128
    yf, cbf, crf = y.astype(f32), cbi.astype(f32), cri.astype(f32)
    a, b = f32(0.34414) * cbf, f32(0.71414) * crf

    def clamp(v):
        return np.clip(np.trunc(v).astype(np.int64), 0, 255)
    # G = Y - (0.34414 Cb' + 0.71414 Cr'): one rounding moved
    assert _wrong(clamp(yf - (a + b)), cube, 1) == 64
    # double-precision constants and arithmetic
    yd = yi.astype(np.float64)
    dbl = np.stack([clamp(yd + 1.402 * cri), clamp(yd - 0.34414 * cbi - 0.71414 * cri), clamp(yd + 1.772 * cbi)], 1)
    assert _wrong(dbl, cube) == 72
    assert _wrong(dbl[:, 1], cube, 1) == 72
    # an integer offset per chroma sample: Y + floor(term), the term rounded as the reference rounds its products
    off = np.stack([yi + np.floor(f32(1.402) * crf), yi + np.floor((-a) - b), yi + np.floor(f32(1.772) * cbf)], 1)
    off = np.clip(off, 0, 255).astype(np.int64)
    assert _wrong(off, cube) == 218
    assert _wrong(off[:, 1], cube, 1) == 218
    # every product contracted into an FMA: no triple changes (computed in C, with fmaf)
    assert _wrong(sp.ycc_cube(fma=True).reshape(-1, 3), cube) == 0
    # out of gamut: a channel's integer outside 0..255 before the clamp, on 76.1 % of the cube
    ch = [np.trunc(v) for v in (yf + f32(1.402) * crf, (yf - a) - b, yf + f32(1.772) * cbf)]
    out = ((ch[0] < 0) | (ch[0] > 255) | (ch[1] < 0) | (ch[1] > 255) | (ch[2] < 0) | (ch[2] > 255)).mean()
    assert round(100 * out, 1) == 76.1, out


def test_dc_sample_is_the_oracles_on_the_whole_sweep():
    """The closed form of a DC-only block's sample against the single-block decode (which also checks that the block
    decodes flat) and the reduced IDCT at n = 4, 2, 1, on every (c0, q0) of the tier C files."""
    c0, q0 = cc.dc_pairs()
    assert c0.size == 255 * 4096 + len(cc.Q_SWEEP) * 65536
    want = cc.dc_sample(c0, q0)
    for n in (8, 4, 2, 1):
        assert np.array_equal(sp.dc_only(c0, q0, n), want), n
    assert (want == 0).any() and (want == 255).any()
    # the int16 wrap of the de-quantisation is reached: a product past 32767 that decodes other than it would unwrapped
    wide = np.abs(c0 * q0) > 32767
    assert wide.any() and (cc.dc_sample(c0[wide], q0[wide]) != np.where(c0[wide] * q0[wide] > 0, 255, 0)).any()


def test_chroma_dc_decodes_to_its_value():
    v = np.arange(256)
    assert np.array_equal(cc.dc_sample(cc.chroma_dc(v), 1), v)
    for n in (8, 4):
        assert np.array_equal(sp.dc_only(cc.chroma_dc(v), 1, n), v)


@pytest.mark.parametrize("n", [8, 4])
def test_library_decodes_partition_0_to_255(n):
    lib, vals = cc.library(n), cc.library_values(n)
    assert lib.shape == (256 // (n * n), 64)
    assert np.array_equal(np.sort(vals.ravel()), np.arange(256))
    for b, v in zip(lib, vals):
        assert np.array_equal(cc.decode_block(b, n), v)
    assert np.abs(lib).max() <= 1023 and np.abs(np.diff(lib[:, 0], append=lib[:1, 0])).max() <= 2047


def test_library_reaches_the_exact_re_evaluation():
    """At least one block of library(8) takes the tensor-core kernel's fast tier and has samples the fast tiers
    re-evaluate exactly, so the cube files run the exact-path patching before the colour step."""
    from tools.make_idct_edges import Tables, classify
    c = classify(Tables(), cc.library(8), np.zeros(4, dtype=np.int64))
    assert c["tc_fast"].all()
    assert (c["tc_fast"] & c["tc"]["flagged"].any(axis=1)).any()
    assert c["cc"]["flagged"].any()


def _triples(case):
    t = (case.yc.astype(np.int64) << 16) | (case.cbc.astype(np.int64) << 8) | case.crc
    return np.bincount(t.ravel(), minlength=1 << 24)


def _check_refbind(case):
    from oracle import refbind
    if refbind.available("std"):                                 # the oracle is the reference here too
        r = refbind.decode(case.jpg, mode=1)
        assert r["rc"] == 0 and np.array_equal(r["rgb"], case.rgb()), case.name


@pytest.mark.parametrize("sampling", ["444", "422", "440", "420", "gray"])
def test_tier_a_file(port, sampling):
    case = cc.tier_a(sampling)
    if sampling != "gray":
        assert (case.g["width"], case.g["height"]) == (4096, 4096)
        assert (_triples(case) == 1).all()
    o = port.decode(case.jpg)
    assert o["rc"] == 0
    assert np.array_equal(o["planes"][0], case.y)
    if case.cb is not None:
        assert np.array_equal(o["planes"][1], case.cb) and np.array_equal(o["planes"][2], case.cr)
    assert np.array_equal(o["rgb"], case.rgb())
    _check_refbind(case)


def test_tier_b_file():
    case = cc.tier_b()
    assert (case.g["width"], case.g["height"]) == (8192, 8192) and case.yc.shape == (4096, 4096)
    assert (_triples(case) == 1).all()
    s = sp.decode_scaled(case.jpg, 1)
    assert s["rc"] == 0
    assert np.array_equal(s["rgb"], case.rgb())


def test_tier_c_files(port):
    files = cc.tier_c()
    assert len(files) == 255 + len(cc.Q_SWEEP) + len(cc.THREE_TABLES) + 2
    seen = set()
    for f in files:
        case = f.case(8)
        o = port.decode(f.jpg)
        assert o["rc"] == 0, f.name
        for got, want in zip(o["planes"], (case.y, case.cb, case.cr)):
            assert want is None or np.array_equal(got, want), f.name
        assert np.array_equal(o["rgb"], case.rgb()), f.name
        if f.name.startswith(("c_gray_q", "c_int16_q")):
            seen |= set(zip(f.c0[0].tolist(), [f.q0[0]] * len(f.c0[0])))
        if f.name.startswith("c_444_three"):
            assert not np.array_equal(cc.dc_sample(f.c0[1], f.q0[1]),
                                      cc.dc_sample(f.c0[1], cc.THREE_TABLES[int(f.name[-1])][1])), f.name
        if f.name.endswith("acwrap"):
            assert (port.decode(f.jpg, entropy_only=True)["coef"][:, 1:] != 0).any(axis=1).all(), f.name
    c0, q0 = cc.dc_pairs()
    assert seen == set(zip(c0.tolist(), q0.tolist()))
