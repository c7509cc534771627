"""Random legal multi-scan scripts and adversarial coefficient arrays, for the multi-scan writer
(tests/multiscan_writer.py) and the reference decoder (tests/t81_decode.py).

random_script() draws a progressive (or, with sequential=True, a non-interleaved sequential) scan script that T.81
G.1.1.1 allows and libjpeg decodes: DC scans over random groups of components, per-component AC bands refined along
sub-ranges that cut across the first-pass bands, positions left uncoded, a DRI per scan and Huffman tables per
scan.  random_coefficients() fills a [blocks, 64] array with blocks from a catalogue of extremes.  random_case()
puts the two together with a baseline template of the same geometry.

TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import io

import numpy as np
from PIL import Image

from tests import multiscan_writer as mw
from tests.jpeg_writer import blocks_to_jpeg

SAMPLINGS = ["gray", "4:4:4", "4:2:2", "4:2:0", "4:4:0"]


def scan_grid(geometry: dict, comps) -> int:
    """MCUs of a scan over `comps` (T.81 A.2): the MCU grid when interleaved or for a 1x1 chroma component, luma's
    own block grid when luma is alone."""
    if len(comps) == 1 and comps[0] == 0 and geometry["ncomp"] == 3:
        return -(-geometry["width"] // 8) * -(-geometry["height"] // 8)
    return geometry["mcus_x"] * geometry["mcus_y"]


def _groups(rng, comps):
    """A random partition of `comps` into groups, each in frame order, the groups in random order."""
    label = rng.integers(0, len(comps), len(comps))
    groups = [tuple(c for c, g in zip(comps, label) if g == k) for k in range(len(comps))]
    groups = [g for g in groups if g]
    rng.shuffle(groups)
    return groups


def _merge(rng, lists, ready):
    """Interleave `lists` at random, keeping the order of each; ready(scan, done) says whether a head may go next."""
    out, heads = [], [0] * len(lists)
    while any(h < len(lst) for h, lst in zip(heads, lists)):
        ok = [i for i, lst in enumerate(lists) if heads[i] < len(lst) and ready(lst[heads[i]], out)]
        i = ok[int(rng.integers(len(ok)))]
        out.append(lists[i][heads[i]])
        heads[i] += 1
    return out


def _ac_scans(rng, c, max_refine, complete):
    """The AC scans of component c: first passes over a random partition of 1..63, then refinements along random
    contiguous ranges of coefficients that share their current Al.  Unless `complete`, some bands are left uncoded
    and refinement sometimes stops before Al 0."""
    if not complete and rng.random() < 0.1:
        return []                                             # this component's AC left uncoded
    cuts = sorted(set(int(x) for x in rng.integers(2, 64, int(rng.integers(0, 6)))))
    edges = [1] + cuts + [64]
    als = [int(rng.integers(0, 14)), int(rng.integers(0, 14))]
    cur = [-1] * 64                                           # current Al per coefficient (-1: uncoded)
    scans = []
    for lo, hi in zip(edges[:-1], edges[1:]):
        if not complete and rng.random() < 0.12:
            continue                                          # a band no scan codes
        al = als[int(rng.integers(2))] if rng.random() < 0.8 else int(rng.integers(0, 14))
        scans.append(((c,), lo, hi - 1, 0, al))
        cur[lo:hi] = [al] * (hi - lo)
    n_refine = int(rng.integers(0, max_refine + 1)) if rng.random() < 0.3 else max_refine
    for _ in range(64 * 14 if complete else n_refine):
        open_ = [k for k in range(1, 64) if cur[k] > 0]
        if not open_:
            break
        k = open_[int(rng.integers(len(open_)))]
        lo = hi = k
        while lo > 1 and cur[lo - 1] == cur[k]:
            lo -= 1
        while hi < 63 and cur[hi + 1] == cur[k]:
            hi += 1
        if rng.random() < 0.5:                                # a sub-range of the run of equal Al
            lo, hi = sorted(int(x) for x in rng.integers(lo, hi + 1, 2))
        al = cur[k]
        scans.append(((c,), lo, hi, al, al - 1))
        cur[lo:hi + 1] = [al - 1] * (hi - lo + 1)
    return scans


def random_script(rng, ncomp: int, geometry: dict, sequential: bool = False, max_scans: int = 256,
                  complete: bool = False):
    """(script, restarts, tables, fill): a legal script [(components, Ss, Se, Ah, Al)] for a frame of `ncomp`
    components, a DRI per scan, a table kind per scan ("flat" / "long" / "mixed") and a fill byte count.
    complete: every coefficient coded down to Al 0.  Otherwise a DC refinement may stop early, but at Al 10 or
    below, so that the DC a decoder holds stays within [-1024, 1023] (an arithmetic shift by 11 or more moves -1
    to -2048)."""
    comps = list(range(ncomp))
    for _ in range(100):
        if sequential:
            script = [(g, 0, 63, 0, 0) for g in _groups(rng, comps)]
        else:
            dc_al = int(rng.integers(0, 14))
            dc_final = 0 if complete or rng.random() < 0.7 else int(rng.integers(0, min(dc_al, 10) + 1))
            dc = [(g, 0, 0, 0, dc_al) for g in _groups(rng, comps)]
            for al in range(dc_al - 1, dc_final - 1, -1):
                dc += [(g, 0, 0, al + 1, al) for g in _groups(rng, comps)]
            ac = [_ac_scans(rng, c, int(rng.integers(0, 20)), complete) for c in comps]

            def ready(scan, done):                            # a component's AC after its DC first pass
                if scan[1] == 0:
                    return True
                return any(s[1] == 0 and s[3] == 0 and scan[0][0] in s[0] for s in done)
            script = _merge(rng, [dc] + ac, ready)
        if len(script) <= max_scans:
            break
    else:
        raise AssertionError("no script within the scan cap")
    restarts = []
    for comps_ in (s[0] for s in script):
        grid = scan_grid(geometry, comps_)
        choice = [0, 1, 2, 3, 7, grid - 1, grid, grid + 5, 65535]
        restarts.append(max(0, min(65535, choice[int(rng.integers(len(choice)))])))
    tables = [["flat", "long", "mixed"][int(rng.integers(3))] for _ in script]
    fill = int(rng.choice([0, 0, 1, 2, 5]))
    return script, restarts, tables, fill


def random_coefficients(rng, geometry: dict, edges=(1, 6, 63)) -> np.ndarray:
    """int16 [blocks, 64] (zig-zag, absolute DC, MCU order): every block one of the catalogue below.  AC within
    +-1023 and DC within [-1024, 1023], what a baseline twin codes with the standard tables."""
    ncomp = geometry["ncomp"]
    bpm = geometry["hf"] * geometry["vf"] + 2 if ncomp == 3 else 1
    n = geometry["mcus_x"] * geometry["mcus_y"] * bpm
    out = np.zeros((n, 64), dtype=np.int64)
    zz = np.arange(64)
    powers = [1, 2, 3, 7, 8, 15, 16, 31, 64, 127, 255, 256, 511, 512, 1023]
    for b in range(n):
        kind = int(rng.integers(8))
        blk = out[b]
        if kind == 0:                                         # DC only
            pass
        elif kind == 1:                                       # photographic: decaying with the zig-zag index
            scale = 400.0 * np.exp(-zz[1:] / rng.uniform(2, 12))
            blk[1:] = np.round(rng.normal(0, 1, 63) * scale * (rng.random(63) < 0.6))
        elif kind == 2:                                       # dense: every AC nonzero
            v = rng.integers(1, 1024, 63) * rng.choice([-1, 1], 63)
            blk[1:] = v
        elif kind == 3:                                       # one coefficient at 1, 63 or a band edge
            k = int(rng.choice(list(edges) + [1, 63]))
            blk[k] = int(rng.choice(powers)) * int(rng.choice([-1, 1]))
        elif kind == 4:                                       # +-1, +-2^j, +-(2^j - 1), +-1023 at random places
            m = rng.random(63) < 0.4
            blk[1:] = np.where(m, rng.choice(powers, 63) * rng.choice([-1, 1], 63), 0)
        elif kind == 5:                                       # alternating +-1
            blk[1:] = np.where(np.arange(63) % 2, -1, 1)
        elif kind == 6:                                       # odd negatives
            blk[1:] = np.where(rng.random(63) < 0.5, -(2 * rng.integers(0, 512, 63) + 1), 0)
        else:                                                 # sparse small values
            blk[1:] = np.where(rng.random(63) < 0.1, rng.integers(-3, 4, 63), 0)
        r = rng.random()
        blk[0] = -1024 if r < 0.15 else 1023 if r < 0.3 else int(rng.integers(-1024, 1024))
    out[:, 1:] = np.clip(out[:, 1:], -1023, 1023)
    # DC -1024 and 1023 side by side: differences of +-2047
    for b in range(0, n - 1, 7):
        out[b, 0], out[b + 1, 0] = -1024, 1023
    # MCU-padding luma blocks: a DC refinement over (0, ...) codes the low bits of their DC even when the first pass
    # over luma alone left it 0, so it stays within [0, 1023] (what the twin can code) only for a DC of 0..1023
    pad = ~mw.coded_mask(geometry)
    out[pad, 0] = np.abs(out[pad, 0]) & 1023
    return out.astype(np.int16)


def template(width: int, height: int, sampling: str) -> bytes:
    """A baseline file of the size and sampling, with libjpeg's standard Huffman tables (what blocks_to_jpeg needs)."""
    rgb = np.full((height, width, 3), 128, np.uint8)
    if sampling == "4:4:0":
        from tests.cases import encode_jpeg_cv
        return encode_jpeg_cv(rgb, 90, "440")
    im = Image.fromarray(rgb)
    kw = dict(format="JPEG", quality=90, optimize=False, progressive=False)
    if sampling == "gray":
        im = im.convert("L")
    else:
        kw["subsampling"] = {"4:4:4": 0, "4:2:2": 1, "4:2:0": 2}[sampling]
    buf = io.BytesIO()
    im.save(buf, **kw)
    return buf.getvalue()


def random_case(seed: int, width: int, height: int, sampling: str, sequential: bool = False, max_scans: int = 256,
                complete: bool = False, port=None):
    """dict(file, twin, script, restarts, tables, fill, coef, expected, geometry) of one random image.  The twin is
    the baseline file of `expected`, the coefficients the script codes."""
    rng = np.random.default_rng(seed)
    tmpl = template(width, height, sampling)
    geometry = port.decode(tmpl, entropy_only=True)["geometry"]
    coef = random_coefficients(rng, geometry)
    ncomp = geometry["ncomp"]
    script, restarts, tables, fill = random_script(rng, ncomp, geometry, sequential, max_scans, complete)
    expected = mw.expected_after(coef, ncomp, geometry, script, len(script))
    quant = {0: rng.integers(1, 17, 64), 1: rng.integers(1, 17, 64)}
    twin = blocks_to_jpeg(tmpl, expected, geometry, quant if ncomp == 3 else {0: quant[0]})
    file = mw.write_multiscan(twin, expected, geometry, script, progressive=not sequential, restarts=restarts,
                              tables=tables, fill=fill, seed=seed)
    return dict(file=file, twin=twin, script=script, restarts=restarts, tables=tables, fill=fill, coef=coef,
                expected=expected, geometry=geometry)


def eob_ladder(geometry: dict, seed: int = 0, corrections: int = 0, rungs: bool = True) -> np.ndarray:
    """int16 [blocks, 64] that is almost all empty AC: DC only, except "rung" blocks placed so that the runs of empty
    blocks between them have lengths 1, 2, 4, ..., up to the last block, so that a scan over one component codes
    EOBn for every n that fits (n = 14 from 16,384 blocks on).  Rung blocks hold 5, 2, 1, -5, -3, -1, ... in every
    AC position: each is nonzero in the first pass at Al 2 and new at the refinements to Al 1 and 0 of libjpeg's
    default script, so it ends the EOB run of every such scan.  With `corrections`, that many blocks (spread
    evenly) hold +-4 in every AC position: inside EOB runs of refinements, each adds 63 correction bits and no new
    coefficient (they hold nothing in 1..5, so that the first pass over 1..5 keeps its long runs).  Without `rungs`
    only block 0 is one."""
    rng = np.random.default_rng(seed)
    ncomp = geometry["ncomp"]
    bpm = geometry["hf"] * geometry["vf"] + 2 if ncomp == 3 else 1
    n = geometry["mcus_x"] * geometry["mcus_y"] * bpm
    out = np.zeros((n, 64), dtype=np.int64)
    out[:, 0] = rng.integers(-1024, 1024, n)
    rung = np.resize(np.array([5, 2, 1, -5, -3, -1]), 63)
    at, gap = 0, 1
    while at < n:
        out[at, 1:] = rung
        at += gap + 1 if rungs else n
        gap *= 2
    for b in np.linspace(1, 0.4 * n, corrections).astype(int) if corrections else []:
        out[b, 1:6] = 0
        out[b, 6:] = np.where(np.arange(58) % 2, 4, -4)
    pad = ~mw.coded_mask(geometry)
    out[pad, 0] = np.abs(out[pad, 0]) & 1023
    return out.astype(np.int16)
