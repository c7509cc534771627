"""Writes multi-scan JPEG files from a coefficient array: non-interleaved sequential files (one SOF0 scan per
component) and progressive files (SOF2) from an explicit scan script.  The input is what
``oracle.port.decode(baseline, entropy_only=True)`` returns for a baseline template file, so every file written
here carries exactly the template's quantised coefficients: the template is its baseline twin.

Every scan gets its own Huffman tables over the symbols it uses, written in a DHT just before its SOS; a DRI can
change between scans.  The code of a scan is one of (never the all-ones code):
  "flat"   up to 128 eight-bit codes, then nine-bit codes
  "long"   every code 11 to 16 bits long, so that every lookup goes through a decoder's second-level table
  "mixed"  random lengths 1 to 16, with one code of each length 11 to 16 whenever there are six or more symbols
Optional 0xFF fill bytes (T.81 B.1.1.2) go before every RSTn and before the marker that follows each scan.

TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import struct

import numpy as np

from tests.jpeg_writer import BitWriter, _seg, block_index, segments

# libjpeg's default progressive script for three components (jcparam.c jpeg_simple_progression):
# (components, Ss, Se, Ah, Al)
DEFAULT_SCRIPT_COLOR = [((0, 1, 2), 0, 0, 0, 1), ((0,), 1, 5, 0, 2), ((2,), 1, 63, 0, 1), ((1,), 1, 63, 0, 1),
                        ((0,), 6, 63, 0, 2), ((0,), 1, 63, 2, 1), ((0, 1, 2), 0, 0, 1, 0), ((2,), 1, 63, 1, 0),
                        ((1,), 1, 63, 1, 0), ((0,), 1, 63, 1, 0)]
DEFAULT_SCRIPT_GRAY = [((0,), 0, 0, 0, 1), ((0,), 1, 5, 0, 2), ((0,), 6, 63, 0, 2), ((0,), 1, 63, 2, 1),
                       ((0,), 0, 0, 1, 0), ((0,), 1, 63, 1, 0)]


def flat_table(symbols) -> tuple[list, list]:
    """(bits[16], vals): the first 128 symbols get 8-bit codes, the rest 9-bit codes (never all ones)."""
    vals = sorted(set(symbols)) or [0]
    assert len(vals) <= 256
    bits = [0] * 16
    bits[7] = min(len(vals), 128)
    bits[8] = len(vals) - bits[7]
    return bits, vals


def long_table(symbols, rng) -> tuple[list, list]:
    """(bits[16], vals): every symbol a code of 11 to 16 bits (at most 256 symbols: the Kraft sum stays below 1/8)."""
    vals = sorted(set(symbols)) or [0]
    return _table_of_lengths(vals, [int(x) for x in rng.integers(11, 17, len(vals))], rng)


def mixed_table(symbols, rng) -> tuple[list, list]:
    """(bits[16], vals): random code lengths 1..16 whose Kraft sum stays below 1 (so the all-ones code is never
    assigned), one symbol at each length 11..16 when there are six or more symbols."""
    vals = sorted(set(symbols)) or [0]
    rng.shuffle(vals)
    lengths = list(range(11, 17)) if len(vals) >= 6 else []
    budget = (1 << 16) - 1 - sum(1 << (16 - L) for L in lengths)        # in units of 2^-16, one code kept free
    for k in range(len(lengths), len(vals)):
        spare = budget - (len(vals) - k - 1)                             # the rest need at least 16-bit codes
        fits = [L for L in range(1, 17) if (1 << (16 - L)) <= spare]
        L = fits[int(rng.integers(len(fits)))]
        lengths.append(L)
        budget -= 1 << (16 - L)
    return _table_of_lengths(vals, lengths, rng)


def _table_of_lengths(vals, lengths, rng):
    order = sorted(range(len(vals)), key=lambda k: (lengths[k], rng.random()))
    bits = [0] * 16
    for L in lengths:
        bits[L - 1] += 1
    return bits, [vals[k] for k in order]


TABLES = {"flat": lambda symbols, rng: flat_table(symbols), "long": long_table, "mixed": mixed_table}


def _codes(bits, vals):
    codes, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            codes[vals[k]] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return codes


class _Geom:
    def __init__(self, g: dict):
        self.g = g
        self.ncomp = g["ncomp"]
        self.hf, self.vf = g["hf"], g["vf"]
        self.mx, self.my = g["mcus_x"], g["mcus_y"]
        self.ny = self.hf * self.vf if self.ncomp == 3 else 1

    def mcus(self, comps):
        """[(component, block row)] per MCU of a scan over `comps`, in scan order."""
        if len(comps) > 1:
            for m in range(self.mx * self.my):
                yield [(c, block_index(self.g, self.ncomp, m, c, s)) for c in comps for s in range(self.ny if c == 0 else 1)]
        else:
            c = comps[0]
            if c == 0 and self.ncomp == 3:
                bw, bh = -(-self.g["width"] // 8), -(-self.g["height"] // 8)
                for by in range(bh):
                    for bx in range(bw):
                        m = (by // self.vf) * self.mx + bx // self.hf
                        yield [(0, block_index(self.g, 3, m, 0, (by % self.vf) * self.hf + bx % self.hf))]
            else:
                for m in range(self.mx * self.my):
                    yield [(c, block_index(self.g, self.ncomp, m, c, 0))]


def _cat(v: int) -> int:
    return abs(v).bit_length()


def _bits_of(v: int, n: int) -> int:
    return v if v >= 0 else v + (1 << n) - 1


class _Scan:
    """Symbols and raw bits of one scan, recorded first (to build its tables), then emitted."""

    def __init__(self):
        self.ops = []           # ("dc" | "ac", symbol) / ("bits", value, n) / ("rst",)

    def sym(self, cls, s):
        self.ops.append((cls, s))

    def bits(self, v, n):
        if n:
            self.ops.append(("bits", v, n))

    def emit(self, table="flat", rng=None, fill=0):
        dc = TABLES[table]([o[1] for o in self.ops if o[0] == "dc"], rng)
        ac = TABLES[table]([o[1] for o in self.ops if o[0] == "ac"], rng)
        cd, ca = _codes(*dc), _codes(*ac)
        out, bw, rst = bytearray(), BitWriter(), 0
        for o in self.ops:
            if o[0] == "dc":
                bw.put(*cd[o[1]])
            elif o[0] == "ac":
                bw.put(*ca[o[1]])
            elif o[0] == "bits":
                bw.put(o[1], o[2])
            else:
                bw.flush()
                out += bw.out + b"\xff" * fill + bytes([0xFF, 0xD0 + (rst & 7)])
                bw, rst = BitWriter(), rst + 1
        bw.flush()
        return bytes(out + bw.out + b"\xff" * fill), dc, ac


def _encode_scan(coef, geo: _Geom, comps, ss, se, ah, al, restart, table="flat", rng=None, fill=0):
    sc = _Scan()
    c64 = np.asarray(coef, dtype=np.int64)
    pred = {c: 0 for c in comps}
    st = dict(eobrun=0, be=[])

    def flush_eob():
        if st["eobrun"]:
            n = st["eobrun"].bit_length() - 1
            sc.sym("ac", n << 4)
            sc.bits(st["eobrun"] - (1 << n), n)
            for b in st["be"]:
                sc.bits(b, 1)
            st["eobrun"], st["be"] = 0, []

    for mi, blocks in enumerate(geo.mcus(comps)):
        if restart and mi and mi % restart == 0:
            flush_eob()
            sc.ops.append(("rst",))
            pred = {c: 0 for c in comps}
        for c, row in blocks:
            blk = c64[row]
            if ss == 0 and se == 63:                            # sequential
                diff = int(blk[0]) - pred[c]
                pred[c] = int(blk[0])
                sc.sym("dc", _cat(diff)); sc.bits(_bits_of(diff, _cat(diff)), _cat(diff))
                r = 0
                nz = np.nonzero(blk[1:])[0]
                last = int(nz[-1]) + 1 if len(nz) else 0
                for k in range(1, last + 1):
                    v = int(blk[k])
                    if v == 0:
                        r += 1
                        continue
                    while r > 15:
                        sc.sym("ac", 0xF0); r -= 16
                    sc.sym("ac", (r << 4) | _cat(v)); sc.bits(_bits_of(v, _cat(v)), _cat(v))
                    r = 0
                if last < 63:
                    sc.sym("ac", 0x00)
            elif ss == 0 and ah == 0:                           # DC first
                v = int(blk[0]) >> al
                diff = v - pred[c]
                pred[c] = v
                sc.sym("dc", _cat(diff)); sc.bits(_bits_of(diff, _cat(diff)), _cat(diff))
            elif ss == 0:                                       # DC refine
                sc.bits((int(blk[0]) >> al) & 1, 1)
            elif ah == 0:                                       # AC first
                if not (np.abs(blk[ss:se + 1]) >> al).any():    # an empty band: only the EOB run grows
                    st["eobrun"] += 1
                    if st["eobrun"] == 0x7FFF:
                        flush_eob()
                    continue
                r = 0
                for k in range(ss, se + 1):
                    v = int(blk[k])
                    a = abs(v) >> al
                    if a == 0:
                        r += 1
                        continue
                    flush_eob()
                    while r > 15:
                        sc.sym("ac", 0xF0); r -= 16
                    n = a.bit_length()
                    sc.sym("ac", (r << 4) | n); sc.bits(a if v > 0 else (~a) & ((1 << n) - 1), n)
                    r = 0
                if r:
                    st["eobrun"] += 1
                    if st["eobrun"] == 0x7FFF:
                        flush_eob()
            else:                                               # AC refine (T.81 G.1.2.3, as libjpeg's encoder)
                if not (np.abs(blk[ss:se + 1]) >> al).any():    # an empty band: only the EOB run grows
                    st["eobrun"] += 1
                    if st["eobrun"] == 0x7FFF:
                        flush_eob()
                    continue
                absv = [abs(int(blk[k])) >> al for k in range(64)]
                eob = max([k for k in range(ss, se + 1) if absv[k] == 1], default=0)
                r, br = 0, []
                for k in range(ss, se + 1):
                    a = absv[k]
                    if a == 0:
                        r += 1
                        continue
                    while r > 15 and k <= eob:
                        flush_eob()
                        sc.sym("ac", 0xF0); r -= 16
                        for b in br:
                            sc.bits(b, 1)
                        br = []
                    if a > 1:
                        br.append(a & 1)
                        continue
                    flush_eob()
                    sc.sym("ac", (r << 4) | 1); sc.bits(0 if blk[k] < 0 else 1, 1)
                    for b in br:
                        sc.bits(b, 1)
                    br, r = [], 0
                if r or br:
                    st["eobrun"] += 1
                    st["be"] += br
                    if st["eobrun"] == 0x7FFF or len(st["be"]) > 937:
                        flush_eob()
    flush_eob()
    return sc.emit(table, rng, fill)


def write_multiscan(template: bytes, coef: np.ndarray, geometry: dict, script, progressive: bool = True,
                    restarts=None, truncate_after: int | None = None, tables="flat", fill: int = 0,
                    seed: int = 0) -> bytes:
    """A multi-scan file with the coefficients `coef` ([blocks, 64] zig-zag, absolute DC, MCU order, as
    port.decode(template, entropy_only=True)["coef"]).  script: [(components, Ss, Se, Ah, Al)], frame component
    indices; restarts: per scan the DRI in that scan's MCUs (0 / None: none); truncate_after: stop (EOI) after
    that many scans; tables: "flat", "long" or "mixed" (see above), for every scan or a list with one per scan;
    fill: 0xFF fill bytes before every RSTn and before the marker after each scan; seed: of the random tables."""
    segs, _ = segments(template)
    geo = _Geom(geometry)
    sof = [p for m, p in segs if m in (0xC0, 0xC1)][0]
    comp_ids = [sof[6 + 3 * c] for c in range(geo.ncomp)]
    out = bytearray(b"\xff\xd8")
    for m, p in segs:
        if m in (0xC4, 0xDA, 0xDD):
            continue
        if m in (0xC0, 0xC1):
            m = 0xC2 if progressive else 0xC0
        out += _seg(m, p)
    dri = None
    for n, (comps, ss, se, ah, al) in enumerate(script):
        if truncate_after is not None and n >= truncate_after:
            break
        ri = (restarts[n] if restarts else 0) or 0
        table = tables if isinstance(tables, str) else tables[n]
        data, dc, ac = _encode_scan(coef, geo, list(comps), ss, se, ah, al, ri, table,
                                    np.random.default_rng([seed, n]), fill)
        # tables for this scan: DC in slot n % 2, AC in slot (n + 1) % 4, so the selectors change between scans
        tdc, tac = n % 2, (n + 1) % 4
        payload = b""
        if ss == 0 and ah == 0:
            payload += bytes([tdc]) + bytes(dc[0]) + bytes(dc[1])
        if se > 0:
            payload += bytes([0x10 | tac]) + bytes(ac[0]) + bytes(ac[1])
        if payload:
            out += _seg(0xC4, payload)
        if ri != dri:
            out += _seg(0xDD, struct.pack(">H", ri))
            dri = ri
        sos = bytes([len(comps)]) + b"".join(bytes([comp_ids[c], (tdc << 4) | tac]) for c in comps)
        out += _seg(0xDA, sos + bytes([ss, se, (ah << 4) | al]))
        out += data
    return bytes(out + b"\xff\xd9")


def write_non_interleaved(template: bytes, coef: np.ndarray, geometry: dict, restart_blocks: int = 0) -> bytes:
    """Sequential (SOF0) file with one scan per component; restart_blocks: DRI in blocks (= MCUs of such a scan)."""
    ncomp = geometry["ncomp"]
    return write_multiscan(template, coef, geometry, [((c,), 0, 63, 0, 0) for c in range(ncomp)], progressive=False,
                           restarts=[restart_blocks] * ncomp)


def coded_mask(geometry: dict) -> np.ndarray:
    """Blocks that hold pixels of the image (the MCU-padding luma blocks of a colour image lie outside luma's own
    block grid: a scan of luma alone does not code them)."""
    ncomp, hf, vf = geometry["ncomp"], geometry["hf"], geometry["vf"]
    ny = hf * vf if ncomp == 3 else 1
    bpm = ny + 2 if ncomp == 3 else 1
    bw, bh = -(-geometry["width"] // 8), -(-geometry["height"] // 8)
    m = np.ones(geometry["mcus_x"] * geometry["mcus_y"] * bpm, dtype=bool)
    if ncomp == 3:
        for mcu in range(geometry["mcus_x"] * geometry["mcus_y"]):
            my, mx = divmod(mcu, geometry["mcus_x"])
            for s in range(ny):
                by, bx = my * vf + s // hf, mx * hf + s % hf
                m[mcu * bpm + s] = by < bh and bx < bw
    return m


def expected_after(coef: np.ndarray, ncomp: int, geometry: dict, script, k: int) -> np.ndarray:
    """The coefficients the first k scans of `script` define (numpy; for files cut after scan k): sign-magnitude
    |v| >> Al for AC first passes, an arithmetic shift for DC, refinement bits added back, whole blocks for sequential
    scans (Ss 0, Se 63).  Positions no scan codes
    are 0, among them the MCU-padding luma blocks of scans over luma alone; a refinement band need not be a band of
    the first passes."""
    c = np.asarray(coef, dtype=np.int32)
    out = np.zeros_like(c)
    ny = geometry["hf"] * geometry["vf"] if ncomp == 3 else 1
    bpm = ny + 2 if ncomp == 3 else 1
    comp_of = np.array([0 if b < ny else b - ny + 1 for b in range(bpm)] * (c.shape[0] // bpm))
    inside = coded_mask(geometry)
    for comps, ss, se, ah, al in script[:k]:
        rows = np.isin(comp_of, comps)
        if len(comps) == 1:
            rows &= inside
        if ss == 0 and se == 63:                        # sequential: the whole block
            out[rows] = c[rows]
        elif ss == 0 and ah:
            out[rows, 0] |= ((c[rows, 0] >> al) & 1) << al
        elif ss == 0:
            out[rows, 0] = (c[rows, 0] >> al) << al
        else:
            band = c[rows][:, ss:se + 1]
            out[np.ix_(rows, np.arange(ss, se + 1))] = np.sign(band) * ((np.abs(band) >> al) << al)
    return out.astype(np.int16)
