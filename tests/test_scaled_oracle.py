"""CPU tests of the reduced-size decode's definition (HJD_FLAG_SCALE_*, include/hjd.h) as its CPU restatement states it.

No reference exists for scaled output, so the restatement (tests/scaled_oracle.c, hjdo_decode_scaled) is pinned three
ways: at shift 0 it is the reference-pinned full decode byte for byte; at shifts 1..3 an independent float32 numpy
restatement, built from the oracle's coefficients and libm's cosf, gives the same bytes; and on smooth images its output
is close to the d x d box average of the full decode, which a transposed or mis-scaled table would not be."""
import ctypes
import ctypes.util
import glob
import os

import numpy as np
import pytest

from tests import jpeg_writer as jw
from tests import scaled_port as sp
from tests.cases import small_cases
from tools.gen_jpegs import encode_jpeg, synth_rgb

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

# loadjpg.cpp:56-66: position in the zig-zag sequence of natural index n
ZIGZAG = np.array([0, 1, 5, 6, 14, 15, 27, 28, 2, 4, 7, 13, 16, 26, 29, 42, 3, 8, 12, 17, 25, 30, 41, 43,
                   9, 11, 18, 24, 31, 40, 44, 53, 10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38, 46, 51, 55, 60,
                   21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63])

_libm = ctypes.CDLL(ctypes.util.find_library("m"))
_libm.cosf.restype = ctypes.c_float
_libm.cosf.argtypes = [ctypes.c_float]
_libm.sqrtf.restype = ctypes.c_float
_libm.sqrtf.argtypes = [ctypes.c_float]


def cos_n(n):
    """cosN[p][k] = cosf(((2p+1) * k * 3.14f) / (float)(2n)), every step in float32, cosf from libm."""
    f32 = np.float32
    out = np.zeros((n, n), dtype=np.float32)
    for p in range(n):
        for k in range(n):
            arg = f32(f32((2 * p + 1) * k) * f32(3.14)) / f32(2 * n)
            out[p, k] = _libm.cosf(float(arg))
    return out


def cc_table():
    c0 = np.float32(1.0) / np.float32(_libm.sqrtf(2.0))
    c = np.array([c0] + [np.float32(1.0)] * 7, dtype=np.float32)
    return (c[:, None] * c[None, :]).astype(np.float32)


def model_blocks(coef, q, n, raw=None):
    """float32 restatement of the reduced IDCT for many blocks: coef int [B, 64] and q [B, 64] in zig-zag order ->
    uint8 [B, n, n] (row y, column x).  raw (int64 [B, n, n]): receives (int)(0.25 * sum) before the int16 wrap."""
    data = (coef.astype(np.int64) * q.astype(np.int64)).astype(np.int16)        # (int16_t)(int)(coef * q)
    nat = data[:, ZIGZAG].astype(np.float32)                                      # natural order, row-major
    cs, cc = cos_n(n), cc_table()
    out = np.zeros((coef.shape[0], n, n), dtype=np.uint8)
    for y in range(n):
        for x in range(n):
            s = np.zeros(coef.shape[0], dtype=np.float32)
            for u in range(n):                                                    # u horizontal, outer
                for v in range(n):
                    s = s + ((cc[u, v] * nat[:, v * 8 + u]) * cs[x, u]) * cs[y, v]
            val = np.trunc(0.25 * s.astype(np.float64)).astype(np.int64)
            if raw is not None:
                raw[:, y, x] = val
            val = val.astype(np.int16)
            val = (val.astype(np.int32) + 128).astype(np.int16)
            out[:, y, x] = np.clip(val, 0, 255)
    return out


def ycc_to_rgb(yc, cb, cr):
    """hjdo_ycc_to_rgb in float32, one rounding per operation."""
    f32 = np.float32
    yf, cbf, crf = yc.astype(np.float32), (cb.astype(np.int32) - 128).astype(np.float32), (cr.astype(np.int32) - 128).astype(np.float32)
    r = yf + f32(1.402) * crf
    g = (yf - f32(0.34414) * cbf) - f32(0.71414) * crf
    b = yf + f32(1.772) * cbf
    return np.stack([np.clip(np.trunc(ch).astype(np.int64), 0, 255) for ch in (r, g, b)], axis=-1).astype(np.uint8)


def quant_tables(jpg):
    """{table id: 64 values, zig-zag} and the table selector of every frame component."""
    segs, _ = jw.segments(jpg)
    q, tq = {}, []
    for m, p in segs:
        if m == 0xDB:
            k = 0
            while k < len(p):
                q[p[k] & 15] = np.frombuffer(p[k + 1:k + 65], dtype=np.uint8).astype(np.int64)
                k += 65
        elif m in (0xC0, 0xC1):
            tq = [p[6 + 3 * c + 2] for c in range(p[5])]
    return q, tq


def model_decode(port, jpg, shift):
    """The scaled decode assembled in numpy from the oracle's entropy-decoded coefficients."""
    o = port.decode(jpg, entropy_only=True)
    g = o["geometry"]
    coef = o["coef"]
    q, tq = quant_tables(jpg)
    n, d = 8 >> shift, 1 << shift
    hf, vf, mx, my = g["hf"], g["vf"], g["mcus_x"], g["mcus_y"]
    ny = hf * vf if g["ncomp"] == 3 else 1
    bpm = ny + 2 if g["ncomp"] == 3 else 1
    blocks = coef.reshape(mx * my, bpm, 64)
    yb = model_blocks(blocks[:, :ny].reshape(-1, 64), np.broadcast_to(q[tq[0]], (mx * my * ny, 64)), n)
    yp = yb.reshape(my, mx, vf, hf, n, n).transpose(0, 2, 4, 1, 3, 5).reshape(my * vf * n, mx * hf * n)
    if g["ncomp"] == 3:
        qc = np.broadcast_to(q[tq[2]], (mx * my, 64))                       # Cb with Cr's table (loadjpg.cpp:984)
        cb = model_blocks(blocks[:, ny], qc, n).reshape(my, mx, n, n).transpose(0, 2, 1, 3).reshape(my * n, mx * n)
        cr = model_blocks(blocks[:, ny + 1], qc, n).reshape(my, mx, n, n).transpose(0, 2, 1, 3).reshape(my * n, mx * n)
        Y, X = np.indices(yp.shape)
        cbp, crp = cb[Y >> (vf - 1), X >> (hf - 1)], cr[Y >> (vf - 1), X >> (hf - 1)]
    else:
        cbp = crp = np.full(yp.shape, 128, dtype=np.uint8)
    ow, oh = -(-g["width"] // d), -(-g["height"] // d)
    return ycc_to_rgb(yp, cbp, crp)[:oh, :ow]


def all_files():
    files = dict(small_cases())
    for p in sorted(glob.glob(os.path.join(GOLDEN, "*.jpg"))):
        files["golden_" + os.path.basename(p)] = open(p, "rb").read()
    return files


FILES = all_files()


def test_tables_are_the_oracles(port):
    c8, cc = port.idct_tables()
    assert np.array_equal(cos_n(8), c8)
    assert np.array_equal(cc_table(), cc)
    assert np.array_equal(cos_n(1), np.ones((1, 1), dtype=np.float32))


@pytest.mark.parametrize("name", sorted(FILES))
def test_shift0_is_the_full_decode(port, name):
    f = FILES[name]
    full = port.decode(f, want_planes=False, want_coef=False)
    s = sp.decode_scaled(f, 0)
    assert s["rc"] == full["rc"]
    assert np.array_equal(s["rgb"], full["rgb"])


@pytest.mark.parametrize("shift", [1, 2, 3])
@pytest.mark.parametrize("name", sorted(FILES))
def test_scaled_decode_matches_the_numpy_model(port, name, shift):
    f = FILES[name]
    s = sp.decode_scaled(f, shift)
    assert s["rc"] == port.decode(f, entropy_only=True)["rc"]
    assert np.array_equal(s["rgb"], model_decode(port, f, shift))


@pytest.mark.parametrize("w,h", [(1, 1), (17, 16), (37, 53), (61, 35), (8, 8), (9, 7), (16, 17)])
@pytest.mark.parametrize("sub", ["4:2:0", "4:4:4", "4:2:2", "gray"])
def test_output_dimensions(port, w, h, sub):
    f = encode_jpeg(synth_rgb(w, h, w + h), 85, gray=True) if sub == "gray" else encode_jpeg(synth_rgb(w, h, w * h), 85, sub)
    for shift in range(4):
        d = 1 << shift
        s = sp.decode_scaled(f, shift)
        assert (s["width"], s["height"]) == (-(-w // d), -(-h // d))
        assert s["rgb"].shape == (-(-h // d), -(-w // d), 3)


# Mean absolute difference between the scaled decode and the d x d box average of the full decode, on smooth images
# (synth_rgb 256x192 at q90).  Observed on the CPU, the largest over seeds 1-3, for 1/2, 1/4, 1/8:
#   4:4:4  1.25  1.00  0.51
#   4:2:2  1.86  2.78  4.21
#   4:2:0  2.52  3.84  5.82
# Subsampled chroma differs more: a scaled chroma block covers twice the output pixels its full-size samples do after
# the box average.  The bounds are the observed values with 50 % margin.  On 4:4:4, the model with cosN transposed is
# 13.5 / 8.9 away and the one with cosN built with /16 is 5.7 / 6.5 away at 1/2 / 1/4.
MAD_BOUND = {"4:4:4": {1: 1.9, 2: 1.5, 3: 0.8}, "4:2:2": {1: 2.8, 2: 4.2, 3: 6.3}, "4:2:0": {1: 3.8, 2: 5.8, 3: 8.7}}


def box_average(rgb, d):
    h, w, _ = rgb.shape
    oh, ow = -(-h // d), -(-w // d)
    pad = np.zeros((oh * d, ow * d, 3), dtype=np.float64)
    cnt = np.zeros((oh * d, ow * d, 1), dtype=np.float64)
    pad[:h, :w] = rgb
    cnt[:h, :w] = 1
    s = pad.reshape(oh, d, ow, d, 3).sum(axis=(1, 3))
    c = cnt.reshape(oh, d, ow, d, 1).sum(axis=(1, 3))
    return s / c


@pytest.mark.parametrize("sub", ["4:2:0", "4:4:4", "4:2:2"])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_scaled_output_is_close_to_the_box_average(port, sub, seed):
    f = encode_jpeg(synth_rgb(256, 192, seed), 90, sub)
    full = port.decode(f, want_planes=False, want_coef=False)["rgb"]
    for shift in (1, 2, 3):
        got = sp.decode_scaled(f, shift)["rgb"].astype(np.float64)
        mad = np.abs(got - box_average(full, 1 << shift)).mean()
        assert mad < MAD_BOUND[sub][shift], (shift, mad)


def test_mis_scaled_tables_are_caught_by_the_box_average(port):
    """The box-average check has teeth: the model with cosN transposed, or built with /16, is far from it."""
    f = encode_jpeg(synth_rgb(256, 192, 1), 90, "4:4:4")
    full = port.decode(f, want_planes=False, want_coef=False)["rgb"]
    global cos_n
    saved = cos_n
    try:
        for bad in (lambda n: saved(n).T.copy(), lambda n: saved(8)[:n, :n].copy()):
            cos_n = bad
            for shift in (1, 2):
                got = model_decode(port, f, shift).astype(np.float64)
                assert np.abs(got - box_average(full, 1 << shift)).mean() > 2 * MAD_BOUND["4:4:4"][shift]
    finally:
        cos_n = saved


def _edges():
    d = np.load(os.path.join(GOLDEN, "idct_edges.npz"))
    return d["coef"].astype(np.int64), d["quant"][d["qidx"]].astype(np.int64), d["label"]


def test_edge_blocks_through_the_scaled_block(port):
    coef, q, label = _edges()
    for n in (8, 4, 2, 1):
        want = model_blocks(coef, q, n)
        got = np.stack([sp.scaled_block(c, qq, n) for c, qq in zip(coef, q)])
        assert np.array_equal(got, want), n
        if n == 8:
            assert np.array_equal(got, np.stack([port.decode_single_block(c, qq) for c, qq in zip(coef, q)]))


def test_edge_blocks_reach_the_clamp_and_the_wrap(port):
    """The near_sat, dc_* and dq_* blocks reach both clamps.  The set stays inside the int16 range, so the wraps come
    from the same blocks pushed past it: DC x 20 wraps the de-quantisation, and top-left coefficients of +-32767 with
    q = 1 wrap (int16)(int)(0.25 * sum) at n = 4."""
    coef, q, label = _edges()
    sel = np.array([lab.startswith(("near_sat", "dc_", "dq_")) for lab in label])
    pushed = coef[sel].copy()
    pushed[:, 0] *= 20
    big = np.zeros((2, 64), dtype=np.int64)
    for v in range(4):
        for u in range(4):
            big[0, ZIGZAG[v * 8 + u]] = 32767
            big[1, ZIGZAG[v * 8 + u]] = -32767 if (u + v) % 2 else 32767
    blocks = np.concatenate([coef[sel], pushed, big])
    qs = np.concatenate([q[sel], q[sel], np.ones((2, 64), dtype=np.int64)])
    assert (np.abs(pushed * q[sel]) > 32767).any()
    for n in (4, 2, 1):
        raw = np.zeros((len(blocks), n, n), dtype=np.int64)
        want = model_blocks(blocks, qs, n, raw)
        got = np.stack([sp.scaled_block(c, qq, n) for c, qq in zip(blocks, qs)])
        assert np.array_equal(got, want), n
        assert (got[:sel.sum()] == 0).any() and (got[:sel.sum()] == 255).any(), n
        if n == 4:                      # at n = 2 four terms of at most 32767 cannot leave the int16 range
            assert (np.abs(raw) > 32767).any(), n
