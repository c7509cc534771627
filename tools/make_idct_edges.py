"""Adversarial coefficient blocks for the two fused IDCT kernels -> tests/golden/idct_edges.npz.

Both kernels compute a fast result per sample and re-evaluate in the reference's own float order only the samples
that lie within an error window of a change of the output byte (csrc/mcu_tc.cuh, csrc/kernels.cu hjd_idct_block).
Random or encoder-written blocks reach the window, the fast tier's preconditions and the DC-only shortcut only by
chance; the blocks written here sit on them on purpose.  Each block is selected by CPU emulations of the kernels'
fast tiers (below) against the reference's order of float32 operations, and carries the label of the property it
was selected for; tests/test_idct_edges.py re-derives every label, tests/test_gpu_edges.py decodes the blocks on
the GPU.

Contents: coef [n, 64] int16 (quantised, zig-zag order, DC absolute), qidx [n] (row of quant), quant [t, 64] uint8
(zig-zag order), label [n] str.  Seeded: running this again writes the same file byte for byte.

    python tools/make_idct_edges.py [--out tests/golden/idct_edges.npz]
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F32, F16 = np.float32, np.float16
ZZ = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
               21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60,
               61, 54, 47, 55, 62, 63])           # natural index of zig-zag position p
UNIT = 2.0 ** -24
TC_WINDOW_UNITS = 20.0                            # HJD_TC_WINDOW_UNITS
CC_WINDOW = F32(1.430511474609375e-06)            # 24 * 2^-24, kernels.cu hjd_idct_block

# quantisation tables of the set (zig-zag order)
Q_ONES = np.ones(64, dtype=np.uint8)
Q_TWOS = np.full(64, 2, dtype=np.uint8)
Q_PRODUCTS = np.ones(64, dtype=np.uint8)          # products at the FP16 limit: DC 3 * 683 = 2049, 89 * 23 = 2047, 128 * 16 = 2048,
Q_PRODUCTS[:7] = [3, 89, 128, 5, 7, 23, 16]       # 5 * 410 = 2050, 7 * 293 = 2051 (FP16: 2052)
Q_STD = np.array([16, 11, 12, 14, 12, 10, 16, 14, 13, 14, 18, 17, 16, 19, 24, 40, 26, 24, 22, 22, 24, 49, 35, 37, 29, 40, 58,
                  51, 61, 60, 57, 51, 56, 55, 64, 72, 92, 78, 64, 68, 87, 69, 55, 56, 80, 109, 81, 87, 95, 98, 103, 104, 103,
                  62, 77, 113, 121, 112, 100, 120, 92, 101, 101, 99], dtype=np.uint8)   # JPEG Annex K luminance, zig-zag
QUANT = np.stack([Q_ONES, Q_TWOS, Q_PRODUCTS, Q_STD])


class Tables:
    """The reference's float32 constants (oracle: libm values of loadjpg.cpp:96-102) and the tensor-core kernel's
    integer matrix pair (read back from the tile image the library builds)."""

    def __init__(self):
        from oracle import port
        import hls_jpeg_decoder_b200 as hjd
        cos, cc = port.idct_tables()
        self.cos = cos.astype(F32)                                   # cos[x][u]
        self.ccn = np.array([cc[n & 7][n >> 3] for n in range(64)], dtype=F32)   # C(u)C(v) at natural n = 8v + u
        s = np.arange(64)
        self.cosx = np.stack([self.cos[s & 7, u] for u in range(8)]).astype(F32)  # [u][sample 8y + x] = cos[x][u]
        self.cosy = np.stack([self.cos[s >> 3, v] for v in range(8)]).astype(F32)
        self.hi, self.lo = hjd.idct_matrix()


def dequant(coef, q):
    """(short)(int)(coef * q) per zig-zag position (loadjpg.cpp:150; the float product is exact here), int64."""
    return (coef.astype(np.int64) * q.astype(np.int64)).astype(np.int16).astype(np.int64)


def finish(val):
    """sat_u8((short)((short)(int)val + 128)), loadjpg.cpp:123-137 / 83-91."""
    iv = np.trunc(val.astype(np.float64)).astype(np.int64).astype(np.int16).astype(np.int64)
    return np.clip((iv + 128).astype(np.int16), 0, 255).astype(np.int64)


def sat_byte(val):
    """The kernels' byte of a sample whose 0.25*sum is `val` (no short wrap: |val| <= A/4 is small where used)."""
    return np.clip(np.trunc(val.astype(np.float64)) + 128, 0, 255).astype(np.int64)


def reference(T, coef, q):
    """0.25 * sum in the reference's order of float32 operations (u outer, v inner, products left to right,
    loadjpg.cpp:112-123) -> (val [n, 64] float32 at sample 8y + x, A = sum |C(u)C(v) v| float64)."""
    dq = dequant(coef, q)
    vn = np.zeros_like(dq)
    vn[:, ZZ] = dq
    bp = (T.ccn[None, :] * vn.astype(F32)).astype(F32)
    s = np.zeros((coef.shape[0], 64), dtype=F32)
    for u in range(8):
        for v in range(8):
            t = (bp[:, 8 * v + u, None] * T.cosx[u][None, :]).astype(F32)
            s = (s + (t * T.cosy[v][None, :]).astype(F32)).astype(F32)
    return (F32(0.25) * s).astype(F32), np.abs(bp).sum(axis=1, dtype=np.float64)


def _words(coef):
    """The 32 words of a block as the kernels load them: zig-zag positions 2i (low half) and 2i + 1 (high half)."""
    c = coef.astype(np.int64) & 0xFFFF
    return c[:, 0::2] | (c[:, 1::2] << 16)


def _fp16_cc():
    """C(u)C(v) rounded UP to FP16 per zig-zag position (hjd_cc_bits): 0 at the DC, 0x39A9 on the first row and
    column, 0x3C00 elsewhere."""
    out = np.zeros(64, dtype=F16)
    for p in range(1, 64):
        n = int(ZZ[p])
        out[p] = np.uint16(0x39A9).view(F16) if ((n & 7) == 0 or (n >> 3) == 0) else F16(1.0)
    return out


def tc_fast_tier(T, coef, q, window_units=TC_WINDOW_UNITS):
    """The tensor-core kernel's decisions and fast result (mcu_tc.cuh:374-421, 439-477), per block:
    dict(h [n, 64] float32, win, a_tot float32, acc [n, 4] float16 (the partial A sums by zig-zag position mod 4),
    all_exact, dc_only, dc_wide bool, dc_byte = the DC-only shortcut's sample, fast = the byte the fast tier stores
    (before re-evaluation), flagged [n, 64] = re-evaluated exactly)."""
    n = coef.shape[0]
    c = coef.astype(np.int64)
    qf = q.astype(np.float64)
    # AC: the offset-binary trick converts c mod 1024 into [-512, 511]; the product rounds to FP16
    x = ((c + 512) % 1024) - 512
    v = (x.astype(np.float64) * qf).astype(F16)
    dc_h = (np.float64(1.0) * c[:, 0].astype(F16).astype(np.float64) * qf[:, 0]).astype(F16)
    v[:, 0] = dc_h
    av = np.abs(v)
    vm = av.max(axis=1).astype(F32)
    cc = _fp16_cc()
    acc = np.zeros((n, 4), dtype=F16)            # a2[(p >> 1) & 1].{lo, hi}[p & 1]: zig-zag position mod 4
    with np.errstate(invalid="ignore", over="ignore"):
        for p in range(64):
            k = p & 3
            acc[:, k] = (av[:, p].astype(np.float64) * np.float64(cc[p]) + acc[:, k].astype(np.float64)).astype(F16)
        s_lo = (acc[:, 0].astype(np.float64) + acc[:, 2].astype(np.float64)).astype(F16)      # __hadd2(a2[0], a2[1])
        s_hi = (acc[:, 1].astype(np.float64) + acc[:, 3].astype(np.float64)).astype(F16)
        a_ac = (s_lo.astype(F32) + s_hi.astype(F32)).astype(F32)
        dc_f = dc_h.astype(F32)
        a_dc = (F32(0.5) * np.abs(dc_f)).astype(F32)
        a_tot = ((a_ac + a_dc).astype(F32) * F32(1.02)).astype(F32)
    w = _words(c)
    chk = np.zeros(n, dtype=np.int64)
    for i in range(1, 32):
        chk |= w[:, i] ^ ((w[:, i] << 1) & 0xFFFFFFFF)
    ac1_bits = w[:, 0] & 0xFFFF0000
    ac1_chk = (w[:, 0] ^ ((w[:, 0] << 1) & 0xFFFFFFFF)) & 0xFC000000
    dc_only = (chk | ac1_bits) == 0
    dc_wide = (c[:, 0] < -2047) | (c[:, 0] > 2047) | ~(vm < 2048)
    with np.errstate(invalid="ignore"):
        all_exact = (~dc_only & ((((chk | ac1_chk) & 0xFC00FC00) != 0) | ~(a_tot < 4000))) | dc_wide
    dc_only = dc_only & ~dc_wide
    win = np.where(dc_only | all_exact, F32(0), (a_tot * F32(window_units * UNIT)).astype(F32)).astype(F32)
    # D = V [M_hi | M_lo]^T is exact (integers); h = D_hi + 2^-24 D_lo in one rounding (the FFMA)
    vz = np.where(all_exact[:, None], 0, v.astype(np.float64))
    d_hi = vz @ T.hi
    d_lo = vz @ T.lo
    h = (d_lo * UNIT + d_hi * 2.0 ** -13).astype(F32)
    p_byte = sat_byte((h + win[:, None]).astype(F32))
    m_byte = sat_byte((h - win[:, None]).astype(F32))
    dc_byte = finish((F32(T.ccn[0]) * dc_f).astype(F32) * F32(0.25))
    fast = np.where(dc_only[:, None], dc_byte[:, None], p_byte)
    flagged = (p_byte != m_byte) & ~dc_only[:, None] | all_exact[:, None]
    return dict(h=h, win=win, a_tot=a_tot, acc=acc, all_exact=all_exact, dc_only=dc_only, dc_wide=dc_wide,
                dc_byte=dc_byte, fast=fast, flagged=flagged, hbyte=sat_byte(h))


def _fma(a, b, c):
    """FP32 FMA as float64 product + sum rounded to FP32 (double rounding is possible but rare)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F32)


def cc_fast_tier(T, coef, q):
    """The CUDA-core kernel's fast result and flags (kernels.cu hjd_idct_block): two FFMA passes on the row pairs
    bp2, pass 1 over u from bp2[vp * 8] (cos[x][0] == 1), pass 2 with 0.25 * cos, h = a2.x + a2.y; re-evaluation
    where |h - rint(h)| <= 24 * 2^-24 * A.  The KM = 20 variant computes the same sums on the blocks it takes
    (the terms it leaves out are zeros), so one emulation serves both.
    dict(h [n, 64], win, fast [n, 64] = byte before re-evaluation, flagged [n, 64])."""
    n = coef.shape[0]
    dq = dequant(coef, q)
    vn = np.zeros_like(dq)
    vn[:, ZZ] = dq
    bp = (T.ccn[None, :] * vn.astype(F32)).astype(F32)
    a_dc = np.abs(bp[:, 0])
    a_ac = np.zeros(n, dtype=F32)
    for p in range(1, 64):
        a_ac = (a_ac + np.abs(bp[:, ZZ[p]])).astype(F32)
    a_tot = (a_ac + a_dc).astype(F32)
    win = np.where(a_ac == 0, F32(-1), (a_tot * CC_WINDOW).astype(F32)).astype(F32)
    cos = T.cos
    r = np.zeros((n, 8, 8), dtype=F32)                       # r[:, v, x]
    for v in range(8):
        acc = np.broadcast_to(bp[:, 8 * v, None], (n, 8)).astype(F32)
        for u in range(1, 8):
            acc = _fma(bp[:, 8 * v + u, None], np.broadcast_to(cos[:, u][None, :], (n, 8)), acc)
        r[:, v, :] = acc
    cq = (F32(0.25) * cos).astype(F32)                       # c_cosq[y * 8 + v]
    h = np.zeros((n, 64), dtype=F32)
    for y in range(8):
        ax = (r[:, 0, :] * cq[y, 0]).astype(F32)
        ay = (r[:, 1, :] * cq[y, 1]).astype(F32)
        for vp in range(1, 4):
            ax = _fma(r[:, 2 * vp, :], np.full((n, 8), cq[y, 2 * vp], dtype=F32), ax)
            ay = _fma(r[:, 2 * vp + 1, :], np.full((n, 8), cq[y, 2 * vp + 1], dtype=F32), ay)
        h[:, 8 * y:8 * y + 8] = (ax + ay).astype(F32)
    hr = ((h + F32(12582912.0)).astype(F32) - F32(12582912.0)).astype(F32)
    d = (h - hr).astype(F32)
    flagged = (np.abs(d) <= win[:, None]) | (a_tot >= F32(1.0e5))[:, None]
    return dict(h=h, win=win, fast=sat_byte(h), flagged=flagged)


def last_index(coef):
    nz = coef[:, 1:] != 0
    return np.where(nz.any(axis=1), 63 - np.argmax(nz[:, ::-1], axis=1), 0)


def near_units(val, A):
    """Distance of every reference sample from the nearest integer, in units of 2^-24 * A."""
    v = val.astype(np.float64)
    return np.abs(v - np.rint(v)) / np.maximum(A * UNIT, 1e-300)[:, None]


def classify(T, coef, qidx):
    """Every property a label can name, per block (bool arrays)."""
    q = QUANT[qidx]
    val, A = reference(T, coef, q)
    ref = finish(val)
    tc = tc_fast_tier(T, coef, q)
    cc = cc_fast_tier(T, coef, q)
    last = last_index(coef)
    tc_fast = ~tc["all_exact"] & ~tc["dc_only"]
    near = near_units(val, A) <= 2.0
    tv = np.trunc(val.astype(np.float64))
    return dict(ref=ref, val=val, A=A, tc=tc, cc=cc, last=last, tc_fast=tc_fast,
                tc_wrong=tc_fast & (tc["hbyte"] != ref).any(axis=1),
                cc_wrong=(cc["fast"] != ref).any(axis=1),
                near=near, near_any=near.any(axis=1) & (A > 0),
                near_sat={t: (near & (tv == t)).any(axis=1) for t in (-129, -128, 127, 128)})


# ---- block generators -------------------------------------------------------------------------------------------

def _dense(rng, n, budget=3000, dc=1016):
    """Dense blocks in [-511, 511] with sum |c| about `budget` (quantised with the all-ones table)."""
    c = np.zeros((n, 64), dtype=np.int64)
    c[:, 0] = rng.integers(-dc, dc + 1, size=n)
    w = rng.exponential(1.0, size=(n, 63)) * (rng.random((n, 63)) < rng.uniform(0.3, 1.0, size=(n, 1)))
    w *= budget / np.maximum(w.sum(axis=1, keepdims=True), 1e-9)
    c[:, 1:] = np.minimum(np.rint(w), 511).astype(np.int64) * rng.choice([-1, 1], size=(n, 63))
    return c


def _short(rng, n, last):
    """Blocks whose last non-zero zig-zag position is `last` (<= 21), fairly large values."""
    c = np.zeros((n, 64), dtype=np.int64)
    c[:, 0] = rng.integers(-1016, 1017, size=n)
    c[:, 1:last + 1] = rng.integers(-400, 401, size=(n, last))
    c[:, last] = rng.integers(1, 400, size=n) * rng.choice([-1, 1], size=n)
    return c


def _column(rng, n):
    """Coefficients in the first column (u = 0) only: the 8 samples of a row are equal, so a row that lands near an
    integer flags 8 samples at once."""
    c = np.zeros((n, 64), dtype=np.int64)
    pos = [int(np.where(ZZ == 8 * v)[0][0]) for v in range(8)]
    c[:, pos[0]] = rng.integers(-1016, 1017, size=n)
    for p in pos[1:]:
        c[:, p] = rng.integers(-511, 512, size=n)
    return c


def _near_sat(rng, n, target):
    """Blocks whose samples sit around `target` (DC ~ 8 * target with the all-ones table) with a moderate AC part."""
    c = np.zeros((n, 64), dtype=np.int64)
    c[:, 0] = 8 * target + 4 + rng.integers(-24, 25, size=n)
    k = rng.integers(3, 12, size=n)
    for i in range(n):
        pos = rng.choice(np.arange(1, 64), size=k[i], replace=False)
        c[i, pos] = rng.integers(-120, 121, size=k[i])
    return c


def _pick(mask, k, rng):
    idx = np.nonzero(mask)[0]
    if len(idx) > k:
        idx = np.sort(rng.choice(idx, size=k, replace=False))
    return idx


def build(seed=20261020):
    T = Tables()
    rng = np.random.default_rng(seed)
    coefs, qids, labels = [], [], []

    def add(c, qi, label):
        c = np.atleast_2d(np.asarray(c, dtype=np.int64))
        coefs.append(c)
        qids.append(np.full(c.shape[0], qi, dtype=np.int64))
        labels.extend([label] * c.shape[0])

    # -- fast tiers wrong, near-integer samples: searched in seeded random pools ---------------------------------
    want = dict(tc_fast_wrong=24, cc_fast_wrong=24, cc_short_fast_wrong=12, near_integer=16)
    got = dict.fromkeys(want, 0)
    for rnd in range(40):
        if all(got[k] >= want[k] for k in want):
            break
        pool = np.concatenate([_dense(rng, 6000, budget=int(b)) for b in (2400, 3000, 3300)] +
                              [_short(rng, 3000, int(last)) for last in (12, 16, 20)])
        qi = np.zeros(pool.shape[0], dtype=np.int64)
        K = classify(T, pool, qi)
        short = K["last"] <= 20
        sel = {"tc_fast_wrong": K["tc_wrong"], "cc_fast_wrong": K["cc_wrong"] & ~short,
               "cc_short_fast_wrong": K["cc_wrong"] & short,
               "near_integer": K["near_any"] & ~K["tc_wrong"] & ~K["cc_wrong"]}
        for name, m in sel.items():
            idx = _pick(m, want[name] - got[name], rng)
            add(pool[idx], 0, name)
            got[name] += len(idx)

    for target, name in ((-129, "near_sat_m129"), (-128, "near_sat_m128"), (127, "near_sat_127"), (128, "near_sat_128")):
        n_got = 0
        for rnd in range(40):
            pool = _near_sat(rng, 8000, target)
            K = classify(T, pool, np.zeros(pool.shape[0], dtype=np.int64))
            idx = _pick(K["near_sat"][target], 4 - n_got, rng)
            add(pool[idx], 0, name)
            n_got += len(idx)
            if n_got >= 4:
                break

    # -- rows of 8 flagged samples (exact-list pressure) -------------------------------------------------------
    pool = _column(rng, 4000)
    tc = tc_fast_tier(T, pool, QUANT[np.zeros(pool.shape[0], dtype=np.int64)])
    rowflags = tc["flagged"].reshape(-1, 8, 8).sum(axis=2).max(axis=1)
    add(pool[_pick((rowflags == 8) & ~tc["all_exact"], 24, rng)], 0, "row_flagged")

    # -- the fast tier's preconditions, each on both sides -----------------------------------------------------
    base = np.zeros(64, dtype=np.int64)
    base[0] = 40
    base[[2, 5, 9]] = [30, -20, 12]
    for pos in (1, 7, 10):                  # position 1 (shares a word with the DC), an odd one, an even one >= 2
        for val, side in ((511, "in"), (-512, "in"), (512, "out"), (-513, "out")):
            c = base.copy()
            c[pos] = val
            add(c, 0, f"ac_range_{side}")
    for pos, cval, side in ((1, 23, "in"), (5, 89, "in"), (2, 16, "out"), (6, 128, "out"), (2, -16, "out"),
                            (3, 410, "out"), (4, 293, "out"), (5, -89, "in"), (2, 15, "in")):
        c = base.copy()
        c[[2, 5]] = 0
        c[pos] = cval                       # de-quantised 2047 | 2048 | 2050 | 2051 with Q_PRODUCTS
        add(c, 2, f"dq_{side}")
    for dc, qi, side in ((2047, 0, "in"), (-2047, 0, "in"), (2048, 0, "out"), (-2048, 0, "out"),
                         (1023, 1, "in"), (1024, 1, "out"), (-1024, 1, "out"), (682, 2, "in"), (683, 2, "out")):
        c = base.copy()
        if qi == 2:
            c[[2, 5]] = 0
        c[0] = dc                           # the quantised DC (all-ones) and the product (x2: 2048; x3: 2049 -> FP16 2048)
        add(c, qi, f"dc_{side}")
    # a_tot on both sides of 4000: one coefficient swept over [0, 511] on dense blocks
    n_a = 0
    for trial in range(200):
        if n_a >= 6:
            break
        b = _dense(rng, 1, budget=int(rng.integers(3400, 3900)))[0]
        pos = int(rng.integers(1, 64))
        sweep = np.repeat(b[None, :], 512, axis=0)
        sweep[:, pos] = np.arange(512) * (1 if b[pos] >= 0 else -1)
        tc = tc_fast_tier(T, sweep, QUANT[np.zeros(512, dtype=np.int64)])
        below = tc["a_tot"] < 4000
        cross = np.nonzero(below[:-1] & ~below[1:])[0]
        if len(cross) == 1 and not tc["all_exact"][cross[0]]:
            add(sweep[cross[0]], 0, "a_below")
            add(sweep[cross[0] + 1], 0, "a_above")
            n_a += 1
    # FP16 A accumulation at its worst: zig-zag positions = 0 (mod 4) -- one of the four half accumulators -- past 2048,
    # then +-1 terms (below half the FP16 spacing there) and 0.7075 terms that round away
    for sgn_pattern in range(4):
        c = np.zeros(64, dtype=np.int64)
        c[0] = int(rng.integers(-200, 201))
        c[[4, 8, 12, 16]] = [511, -511, 511, 511]
        c[24] = 60 + 10 * sgn_pattern
        ones = [p for p in range(28, 64, 4)]
        c[ones] = rng.choice([-1, 1], size=len(ones))
        for p in range(21, 64, 4):          # 0.7075 terms in a second accumulator
            if (ZZ[p] & 7) == 0 or (ZZ[p] >> 3) == 0:
                c[p] = 1
        c[[1, 5, 9, 13]] = [300, 300, -300, 300] if sgn_pattern & 1 else [0, 0, 0, 0]
        add(c, 0, "a_fp16_worst")

    # -- DC-only shortcut and its neighbours -------------------------------------------------------------------
    for dc in (0, 1, -1, 7, -8, 509, -510, 1016, -1024, 2047, -2047):
        c = np.zeros(64, dtype=np.int64)
        c[0] = dc
        add(c, 0, "dc_only")
    for dc, qi in ((1024, 1), (-1024, 1), (683, 2), (2048, 0), (-2048, 0), (1000, 3)):
        c = np.zeros(64, dtype=np.int64)
        c[0] = dc                           # 1000 * 16 = 16000: wraps nothing, far beyond FP16's exact range
        add(c, qi, "dc_only_wide")
    for dc in (0, 300, -300):
        for pos, val in ((1, 1), (1, -1), (63, 1), (63, -1)):
            c = np.zeros(64, dtype=np.int64)
            c[0], c[pos] = dc, val
            add(c, 0, f"dc_plus_{pos}")

    # -- short-block switch: last coefficient at zig-zag 20 (low half of word 10) or 21 (high half) ------------
    for last in (20, 21):
        add(_short(rng, 8, last), 0, f"last_{last}")
        add(_short(rng, 4, last), 3, f"last_{last}")

    coef = np.concatenate(coefs).astype(np.int16)
    qidx = np.concatenate(qids).astype(np.uint8)
    return dict(coef=coef, qidx=qidx, quant=QUANT.astype(np.uint8), label=np.array(labels))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "idct_edges.npz"))
    a = ap.parse_args()
    d = build()
    np.savez_compressed(a.out, **d)
    names, counts = np.unique(d["label"], return_counts=True)
    for nm, k in zip(names, counts):
        print(f"{nm:22s} {k}")
    print(f"{len(d['label'])} blocks -> {a.out} ({os.path.getsize(a.out)} bytes)")


if __name__ == "__main__":
    main()
