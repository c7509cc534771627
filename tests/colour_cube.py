"""Builders for the colour-cube and DC-only tests -- TEST INFRASTRUCTURE ONLY.

The colour step maps one (Y, Cb, Cr) byte triple to three bytes, so its whole input space is 2^24 triples; a DC-only
block decodes to one flat sample that depends on the pair (quantised DC c0, table entry q0) alone.  This module builds
files that hold every triple exactly once, and files that sweep (c0, q0), together with their expected decodes:

- tier A: one 4096 x 4096 file per sampling (4:4:4, 4:2:2, 4:4:0, 4:2:0) whose luma blocks cycle through
  library(8) (four blocks whose 8 x 8 decodes hold each value 0..255 once) and whose chroma blocks are flat DC-only
  blocks, each (Cb, Cr) pair held by the MCUs of one set of four luma blocks; plus a small gray file;
- tier B: one 8192 x 8192 4:2:0 file whose luma blocks cycle through library(4) (sixteen blocks whose reduced 4 x 4
  decodes hold each value once), so that the 1/2-scale decode holds the whole cube;
- tier C: gray and 4:4:4 files with one DC-only block per MCU: every c0 in [-2048, 2047] for every q0 in 1..255, every
  c0 of the int16 range for a few q0, three distinct tables in Y, Cb and Cr, and blocks whose AC coefficients
  de-quantise to 0 through the int16 wrap.

The oracle (oracle/jpeg_oracle.c, through tests/scaled_oracle.c) pins every expectation: ycc_to_rgb against
hjdo_ycc_to_rgb on the whole cube, dc_sample against the single-block decode and the reduced IDCT on the whole sweep,
and each file's decode against its constructed expectation (tests/test_colour_cube.py)."""
from __future__ import annotations

import hashlib
import os

import numpy as np

from tests import jpeg_writer as jw
from tests import scaled_port as sp
from tools.make_idct_edges import ZZ

F32 = np.float32
SAMPLINGS = {"444": (1, 1), "422": (2, 1), "440": (1, 2), "420": (2, 2)}     # luma (hf, vf); chroma 1 x 1
Q_SWEEP = [1, 2, 3, 8, 16, 64, 128, 255]                                      # q0 of the int16-range sweep
THREE_TABLES = [(5, 200, 13), (255, 1, 37), (64, 9, 128)]                   # DC entries of Y, Cb and Cr tables


def ycc_to_rgb(yc, cb, cr):
    """hjdo_ycc_to_rgb in float32, one rounding per operation."""
    f32 = np.float32
    yf, cbf, crf = yc.astype(np.float32), (cb.astype(np.int32) - 128).astype(np.float32), (cr.astype(np.int32) - 128).astype(np.float32)
    r = yf + f32(1.402) * crf
    g = (yf - f32(0.34414) * cbf) - f32(0.71414) * crf
    b = yf + f32(1.772) * cbf
    return np.stack([np.clip(np.trunc(ch).astype(np.int64), 0, 255) for ch in (r, g, b)], axis=-1).astype(np.uint8)


def cube_triples():
    """(Y, Cb, Cr) uint8 arrays of all 2^24 triples, in the order of scaled_port.ycc_cube: index (Y << 16) | (Cb << 8) | Cr."""
    t = np.arange(1 << 24, dtype=np.uint32)
    return (t >> 16).astype(np.uint8), ((t >> 8) & 255).astype(np.uint8), (t & 255).astype(np.uint8)


# ---- DC-only blocks ---------------------------------------------------------------------------------------------

def dc_sample(c0, q0):
    """The flat sample of a DC-only block: the reference's steps with every AC term zero (loadjpg.cpp:150, 120-137,
    83-91): (short)(int)(c0 * q0), times C(0)C(0) in float32, 0.25 * that truncated, the int16 wraps, the clamp."""
    from oracle import port
    cc00 = port.idct_tables()[1][0, 0]
    data = (np.asarray(c0, dtype=np.int64) * np.asarray(q0, dtype=np.int64)).astype(np.int16)
    s = (F32(cc00) * data.astype(F32)).astype(F32)
    val = np.trunc(0.25 * s.astype(np.float64)).astype(np.int64).astype(np.int16)
    return np.clip((val.astype(np.int32) + 128).astype(np.int16), 0, 255).astype(np.uint8)


def chroma_dc(v):
    """The quantised DC that decodes to the flat value v (0..255) with q0 = 1: +-(8 |v - 128| + 1), the sign of v - 128."""
    d = np.asarray(v, dtype=np.int64) - 128
    return np.where(d < 0, -1, 1) * (8 * np.abs(d) + 1)


def dc_cycle():
    """Every c0 in [-2048, 2047] once, in a cyclic order whose steps are 1 or 2: 2047, 2045, ..., -2047, then
    -2048, -2046, ..., 2046.  Any rotation that does not start at -2048 is a valid DC sequence for the standard
    tables (differences within category 11)."""
    return np.concatenate([np.arange(2047, -2048, -2), np.arange(-2048, 2047, 2)])


def int16_sweep():
    """Every c0 of the int16 range: 0, 1, ..., 32767, -32768, ..., -1 (written with dc_mod16: every step is +1)."""
    return np.arange(1 << 16, dtype=np.int64).astype(np.int16).astype(np.int64)


def dc_pairs():
    """(c0, q0) of the whole DC sweep of the tier C files: [-2048, 2047] x 1..255, then the int16 range x Q_SWEEP."""
    c = np.arange(-2048, 2048)
    c0 = [np.tile(c, 255), np.tile(int16_sweep(), len(Q_SWEEP))]
    q0 = [np.repeat(np.arange(1, 256), c.size), np.repeat(Q_SWEEP, 1 << 16)]
    return np.concatenate(c0), np.concatenate(q0)


# ---- luma library -----------------------------------------------------------------------------------------------

def _synthesis(n):
    """[n*n samples (y, x), n*n coefficients (v, u)]: 0.25 * C(u)C(v) cos[x][u] cos[y][v] of the n-point decode, with the
    oracle's cos((2p+1) k 3.14 / 2n) (float64 here: the construction only has to land inside the intervals)."""
    k = np.arange(n)
    cos = np.cos(np.outer(2 * k + 1, k) * 3.14 / (2 * n))                       # cos[p][k]
    c = np.where(k == 0, 1 / np.sqrt(2), 1.0)
    a = 0.25 * np.einsum("u,v,xu,yv->yxvu", c, c, cos, cos)
    return a.reshape(n * n, n * n)


def decode_block(coef, n):
    """One all-ones-table block through the oracle: the single-block decode (n = 8) or the reduced IDCT (n = 4)."""
    from oracle import port
    q = np.ones(64)
    return port.decode_single_block(coef, q) if n == 8 else sp.scaled_block(coef, q, n)


def library(n):
    """Blocks (int64 [256 / n^2, 64], zig-zag, quantisation table all ones) whose n x n decodes hold each
    value 0..255 once: block k decodes to the raster ramp 64k + 8y + x (n = 8, 4 blocks) or 16k + 4y + x (n = 4, 16
    blocks).  Each is the inverse of the decode's transform applied to the ramp shifted to the centre of every
    sample's truncation interval (t - 128, half a unit away from zero), rounded."""
    a = _synthesis(n)
    out = []
    for k in range(256 // (n * n)):
        t = k * n * n + np.arange(n * n)
        s = (t - 128) + 0.5 * np.sign(t - 128)
        f = np.rint(np.linalg.solve(a, s)).astype(np.int64)                      # natural (v, u), n x n
        nat = np.zeros((8, 8), dtype=np.int64)
        nat[:n, :n] = f.reshape(n, n)
        out.append(nat.reshape(64)[ZZ])
    out = np.array(out)
    if n == 8:
        # One +-1 pair found by a seeded search: it keeps block 2's decode and puts one of its samples within the error
        # windows of both fused kernels' fast tiers (tools/make_idct_edges.classify), so that their exact re-evaluation
        # runs on the cube files before the colour step.
        out[2, [21, 37]] += [1, -1]
    return out


def library_values(n):
    """uint8 [blocks, n, n]: what each library(n) block decodes to."""
    return (np.arange(256).reshape(-1, n, n)).astype(np.uint8)


# ---- files ------------------------------------------------------------------------------------------------------

def _template(sampling, w, h):
    """A baseline file with the standard Huffman tables, of sampling "444", "422", "440", "420" or "gray", whose frame
    header states w x h (the scan is a small image's: blocks_to_jpeg replaces it)."""
    from tests import cases
    from tools.gen_jpegs import encode_jpeg, synth_rgb
    px = synth_rgb(16, 16, 1)
    if sampling == "gray":
        t = encode_jpeg(px, 75, gray=True)
    elif sampling == "440":
        t = cases.encode_jpeg_cv(px, 75, "440")
    else:
        t = encode_jpeg(px, 75, {"444": "4:4:4", "422": "4:2:2", "420": "4:2:0"}[sampling])
    segs, _ = jw.segments(t)
    out = bytearray(b"\xff\xd8")
    for m, p in segs:
        if m in (0xC0, 0xC1):
            p = p[:1] + h.to_bytes(2, "big") + w.to_bytes(2, "big") + p[5:]
        out += bytes([0xFF, m]) + (len(p) + 2).to_bytes(2, "big") + p
    return bytes(out) + b"\x00\xff\xd9"


def _geometry(jpg):
    from oracle import port
    return port.info(jpg)


def _luma_plane(values, g, n):
    """Blocks' n x n samples (uint8 [luma blocks in scan order, n, n]) arranged as the luma plane of geometry g."""
    hf, vf = (g["hf"], g["vf"]) if g["ncomp"] == 3 else (1, 1)
    my, mx = g["mcus_y"], g["mcus_x"]
    return values.reshape(my, mx, vf, hf, n, n).transpose(0, 2, 4, 1, 3, 5).reshape(my * vf * n, mx * hf * n)


def _chroma_plane(values, g, n):
    """One value per MCU (uint8 [MCUs]) as a flat n x n tile per MCU: a chroma plane."""
    return np.kron(values.reshape(g["mcus_y"], g["mcus_x"]), np.ones((n, n), dtype=np.uint8))


def upsample(c, g):
    """A chroma plane replicated to the luma plane's size (flat chroma blocks: any replication rule gives this)."""
    hf, vf = (g["hf"], g["vf"]) if g["ncomp"] == 3 else (1, 1)
    return np.repeat(np.repeat(c, vf, axis=0), hf, axis=1)


class Case:
    """A file and its expected decode at 1 / d: planes (Y, and for colour files Cb, Cr: uint8, MCU-padded, in the
    layout of the oracle's and KEEP_PLANES' planes) and rgb (uint8 [ceil(H/d), ceil(W/d), 3])."""

    def __init__(self, name, jpg, y, cb=None, cr=None, d=1):
        self.name, self.jpg, self.d = name, jpg, d
        self.g = _geometry(jpg)
        self.y, self.cb, self.cr = y, cb, cr
        h, w = -(-self.g["height"] // d), -(-self.g["width"] // d)
        if cb is None:
            c = np.full(y.shape, 128, dtype=np.uint8)
            self.cbu = self.cru = c
        else:
            self.cbu, self.cru = upsample(cb, self.g), upsample(cr, self.g)
        self.yc, self.cbc, self.crc = y[:h, :w], self.cbu[:h, :w], self.cru[:h, :w]

    def rgb(self):
        return ycc_to_rgb(self.yc, self.cbc, self.crc)


def _cache_key():
    """Files are cached by name plus a digest of the sources that write them."""
    h = hashlib.sha256()
    here = os.path.dirname(os.path.abspath(__file__))
    for f in ("colour_cube.py", "jpeg_writer.py"):
        with open(os.path.join(here, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:12]


def _cached(name, make):
    from tests.test_gpu_configs import _cached as cached
    return cached(f"colour_{name}_{_cache_key()}", make)


ONES = np.ones(64, dtype=np.uint8)


def tier_a(sampling):
    """4096 x 4096 file of the sampling (or a 32 x 16 gray file): every (Y, Cb, Cr) triple exactly once."""
    if sampling == "gray":
        w, h = 32, 16
        t = _template("gray", w, h)
        g = _geometry(t)
        j = np.arange(g["blocks"]) % 4
        coef = library(8)[j]
        jpg = _cached("a_gray", lambda: jw.blocks_to_jpeg(t, coef, g, {0: ONES}))
        return Case("a_gray", jpg, _luma_plane(library_values(8)[j], g, 8))
    hf, vf = SAMPLINGS[sampling]
    ny, per = hf * vf, 4 // (hf * vf)                 # luma blocks per MCU, MCUs per (Cb, Cr) pair
    t = _template(sampling, 4096, 4096)
    g = _geometry(t)
    n_mcu = g["mcus_x"] * g["mcus_y"]
    assert n_mcu == 65536 * per
    j = np.arange(n_mcu * ny) % 4
    pair = np.arange(n_mcu) // per
    cb, cr = (pair >> 8).astype(np.uint8), (pair & 255).astype(np.uint8)

    def make():
        coef = np.zeros((n_mcu, ny + 2, 64), dtype=np.int64)
        coef[:, :ny] = library(8)[j].reshape(n_mcu, ny, 64)
        coef[:, ny, 0], coef[:, ny + 1, 0] = chroma_dc(cb), chroma_dc(cr)
        return jw.blocks_to_jpeg(t, coef.reshape(-1, 64), g, {0: ONES}, tq=[0, 0, 0])
    jpg = _cached(f"a_{sampling}", make)
    return Case(f"a_{sampling}", jpg, _luma_plane(library_values(8)[j], g, 8), _chroma_plane(cb, g, 8),
                _chroma_plane(cr, g, 8))


def tier_b():
    """8192 x 8192 4:2:0 file whose 1/2-scale decode holds every triple exactly once (Case at d = 2)."""
    t = _template("420", 8192, 8192)
    g = _geometry(t)
    n_mcu = g["mcus_x"] * g["mcus_y"]
    assert n_mcu == 65536 * 4
    j = np.arange(n_mcu * 4) % 16
    pair = np.arange(n_mcu) // 4
    cb, cr = (pair >> 8).astype(np.uint8), (pair & 255).astype(np.uint8)

    def make():
        coef = np.zeros((n_mcu, 6, 64), dtype=np.int64)
        coef[:, :4] = library(4)[j].reshape(n_mcu, 4, 64)
        coef[:, 4, 0], coef[:, 5, 0] = chroma_dc(cb), chroma_dc(cr)
        return jw.blocks_to_jpeg(t, coef.reshape(-1, 64), g, {0: ONES}, tq=[0, 0, 0])
    jpg = _cached("b_420", make)
    return Case("b_420", jpg, _luma_plane(library_values(4)[j], g, 4), _chroma_plane(cb, g, 4),
                _chroma_plane(cr, g, 4), d=2)


def _dc_table(q0, ac=1):
    q = np.full(64, ac, dtype=np.uint8)
    q[0] = q0
    return q


class DcCase:
    """A tier C file: its DC per block (c0 [components][MCUs]) and the q0 each component is de-quantised with."""

    def __init__(self, name, jpg, c0, q0):
        self.name, self.jpg, self.c0, self.q0 = name, jpg, c0, q0
        self.g = _geometry(jpg)

    def case(self, n):
        """The expected decode with n x n samples per block (n = 8 >> shift) as a Case."""
        s = [dc_sample(c, q) for c, q in zip(self.c0, self.q0)]
        planes = [_chroma_plane(v, self.g, n) for v in s]
        return Case(self.name, self.jpg, *planes, d=8 // n)


def tier_c():
    """The DC sweep files (DcCase list)."""
    cyc = dc_cycle()
    out = []
    t = _template("gray", 512, 512)
    g = _geometry(t)
    for q0 in range(1, 256):
        c0 = np.roll(cyc, -(q0 * 17) % 2048)          # rotations that never start at -2048 (index 2048)
        jpg = _cached(f"c_gray_q{q0}", lambda: jw.blocks_to_jpeg(t, _dc_blocks(c0), g, {0: _dc_table(q0)}))
        out.append(DcCase(f"c_gray_q{q0}", jpg, [c0], [q0]))
    t = _template("gray", 2048, 2048)
    g = _geometry(t)
    c0 = int16_sweep()
    for q0 in Q_SWEEP:
        jpg = _cached(f"c_int16_q{q0}", lambda: jw.blocks_to_jpeg(t, _dc_blocks(c0), g, {0: _dc_table(q0)},
                                                                   dc_mod16=True))
        out.append(DcCase(f"c_int16_q{q0}", jpg, [c0], [q0]))
    t = _template("444", 512, 512)
    g = _geometry(t)
    for k, qs in enumerate(THREE_TABLES):             # Cb is de-quantised with Cr's table (loadjpg.cpp:984)
        cs = [np.roll(cyc, -r) for r in (0, 1365, 2730)]
        coef = np.stack([_dc_blocks(c) for c in cs], axis=1).reshape(-1, 64)
        jpg = _cached(f"c_444_three_{k}", lambda: jw.blocks_to_jpeg(
            t, coef, g, {i: _dc_table(q) for i, q in enumerate(qs)}, tq=[0, 1, 2]))
        out.append(DcCase(f"c_444_three_{k}", jpg, cs, [qs[0], qs[2], qs[2]]))
    # AC coefficients of +-512 at q = 128: 512 * 128 = 2^16 de-quantises to 0 through the int16 wrap, so every block
    # decodes as a DC-only block although its coded AC is not zero
    for s in ("gray", "444"):
        t = _template(s, 64, 64)
        g = _geometry(t)
        nb = g["mcus_x"] * g["mcus_y"]
        c0 = (np.arange(nb) * 97) % 2001 - 1000
        blocks = _dc_blocks(c0)
        for i in range(nb):
            if i % 2:
                blocks[i, 1:] = 512 * np.where(np.arange(63) % 3 == 0, -1, 1)
            else:
                blocks[i, 1 + (i * 5) % 63] = -512 if i % 4 else 512
        ncomp = 1 if s == "gray" else 3
        coef = np.repeat(blocks, ncomp, axis=0)
        jpg = _cached(f"c_{s}_acwrap", lambda: jw.blocks_to_jpeg(t, coef, g, {0: _dc_table(3, 128)},
                                                                tq=[0] * ncomp))
        out.append(DcCase(f"c_{s}_acwrap", jpg, [c0] * ncomp, [3] * ncomp))
    return out


def _dc_blocks(c0):
    b = np.zeros((len(c0), 64), dtype=np.int64)
    b[:, 0] = c0
    return b
