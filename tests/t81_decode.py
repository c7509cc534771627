"""A plain reference decoder for multi-scan JPEG files: sequential (SOF0/SOF1, any grouping of components into scans)
and progressive (SOF2) Huffman files, restated from ITU-T T.81 (Annex A.2 for the block grids, Annex B for the
markers, Annex F.2.2 for sequential decoding, Annex G.2 for the progressive procedures; the decode_mcu_* routines of
libjpeg's jdphuff.c follow the same structure).  It decodes entropy-coded data only, and returns the coefficients in
the layout the GPU slab and oracle.port.decode(..., entropy_only=True)["coef"] use: int16 [blocks, 64], MCU order,
the luma blocks of an MCU in raster order then Cb then Cr, zig-zag order, absolute DC.  Positions that no scan codes
are 0.

It imports nothing from the product, the oracle or the test writers, so that it can check all three.

Sequential scans follow plain T.81 F.2.2.2: an AC symbol of size 0 is EOB (run 0) or ZRL (run 15).  The reference
decoder the product reproduces treats the other size-0 symbols differently (it ignores them); no file built by the
test writers contains one, so that quirk is not modelled here.

decode() also returns a coverage record, so that a test can prove which branches a file reaches:
  code_lengths     {kind: set of Huffman code lengths decoded}, kind in "seq_dc" and "seq_ac" (the DC and AC codes
                   of sequential scans), "dc_first", "ac_first", "ac_refine"
  seq_ac_nonzero   nonzero AC coefficients decoded by sequential scans
  seq_zrl          ZRL symbols decoded by sequential scans
  eobn             {"ac_first" / "ac_refine": set of n of the EOBn symbols decoded}
  max_eob_corrections  the most correction bits read inside one EOB run of an AC refinement scan
  fill_bytes       0xFF fill bytes before markers (T.81 B.1.1.2), inside and between entropy-coded segments
  scan_comps       the component tuple (frame indices) of every scan, in file order
  al               {kind: set of Al values}
  levels           the length of the longest chain of scans in which each one codes a (component, coefficient)
                   position that the one before it coded: scans in one chain cannot run at the same time

TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import struct

import numpy as np


class T81Error(ValueError):
    pass


def _huff(bits, vals):
    """T.81 C.2 / F.2.2.3: per length L, (mincode, maxcode, first value index), or None if no code has length L."""
    out, code, k = [None] * 17, 0, 0
    for length in range(1, 17):
        n = bits[length - 1]
        if n:
            out[length] = (code, code + n - 1, k)
        code = (code + n) << 1
        k += n
    return out, list(vals)


class _Bits:
    """Bit reader over the un-stuffed bytes of one restart interval; zero bits past its end."""

    def __init__(self, data: bytes):
        self.d = data + b"\x00" * 8
        self.n = len(data) * 8
        self.p = 0

    def peek16(self) -> int:
        q = self.p >> 3
        if q + 4 > len(self.d):
            self.d += b"\x00" * 8
        return (int.from_bytes(self.d[q:q + 4], "big") >> (16 - (self.p & 7))) & 0xFFFF

    def get(self, n: int) -> int:
        if n == 0:
            return 0
        v = self.peek16() >> (16 - n)           # n <= 16
        self.p += n
        return v

    def decode(self, table, lengths: set) -> int:
        """DECODE of T.81 F.2.2.3, one code length at a time."""
        spec, vals = table
        w = self.peek16()
        for length in range(1, 17):
            code = w >> (16 - length)
            s = spec[length]
            if s is not None and code <= s[1]:
                if code < s[0]:
                    break
                self.p += length
                lengths.add(length)
                return vals[s[2] + code - s[0]]
        raise T81Error("no Huffman code matches")


def _extend(v: int, t: int) -> int:
    """EXTEND of T.81 F.2.2.1."""
    return v - (1 << t) + 1 if t and v < (1 << (t - 1)) else v


def _segment(buf: bytes, i: int, cov: dict):
    """The entropy-coded segment at i: its restart intervals (un-stuffed, with their RSTn numbers) and the offset of
    the marker that ends it.  Fill bytes (0xFF before a marker) are counted and dropped."""
    intervals, cur, rst = [], bytearray(), None
    n = len(buf)
    while i < n:
        b = buf[i]
        if b != 0xFF:
            cur.append(b)
            i += 1
            continue
        j = i + 1
        while j < n and buf[j] == 0xFF:
            j += 1
        if j >= n:
            cov["fill_bytes"] += j - i - 1
            i = n
            break
        m = buf[j]
        if m == 0x00:
            if j != i + 1:
                raise T81Error("fill bytes before a stuffed zero")
            cur.append(0xFF)
            i = j + 1
            continue
        cov["fill_bytes"] += j - i - 1
        if 0xD0 <= m <= 0xD7:
            intervals.append((bytes(cur), rst))
            cur, rst = bytearray(), m - 0xD0
            i = j + 1
            continue
        i = j - 1                               # at the 0xFF of the marker itself
        break
    intervals.append((bytes(cur), rst))
    return intervals, i


class _Frame:
    def __init__(self, payload: bytes, progressive: bool):
        self.progressive = progressive
        if payload[0] != 8:
            raise T81Error("only 8-bit samples")
        self.height, self.width = struct.unpack(">HH", payload[1:5])
        self.ncomp = payload[5]
        self.ids, self.h, self.v = [], [], []
        for c in range(self.ncomp):
            cid, hv = payload[6 + 3 * c], payload[7 + 3 * c]
            self.ids.append(cid)
            self.h.append(hv >> 4)
            self.v.append(hv & 15)
        self.hmax, self.vmax = max(self.h), max(self.v)
        if self.ncomp == 1:                      # one component: an MCU is one block whatever its factors (A.2.2)
            self.h, self.v, self.hmax, self.vmax = [1], [1], 1, 1
        self.mcus_x = -(-self.width // (8 * self.hmax))
        self.mcus_y = -(-self.height // (8 * self.vmax))
        self.offset = np.cumsum([0] + [self.h[c] * self.v[c] for c in range(self.ncomp)]).tolist()
        self.bpm = self.offset[-1]

    def comp_grid(self, c: int):
        """Blocks of component c alone (T.81 A.2.1): ceil(ceil(X * Hc / Hmax) / 8) by ceil(ceil(Y * Vc / Vmax) / 8)."""
        xc = -(-self.width * self.h[c] // self.hmax)
        yc = -(-self.height * self.v[c] // self.vmax)
        return -(-xc // 8), -(-yc // 8)

    def slab_row(self, c: int, bx: int, by: int) -> int:
        mcu = (by // self.v[c]) * self.mcus_x + bx // self.h[c]
        return mcu * self.bpm + self.offset[c] + (by % self.v[c]) * self.h[c] + bx % self.h[c]

    def scan_mcus(self, comps):
        """Per MCU of a scan over `comps`: [(scan component index, slab row)] in coding order (A.2.2, A.2.3)."""
        if len(comps) == 1:
            c = comps[0]
            bw, bh = self.comp_grid(c)
            return [[(0, self.slab_row(c, bx, by))] for by in range(bh) for bx in range(bw)]
        out = []
        for my in range(self.mcus_y):
            for mx in range(self.mcus_x):
                blocks = []
                for k, c in enumerate(comps):
                    for v in range(self.v[c]):
                        for h in range(self.h[c]):
                            blocks.append((k, self.slab_row(c, mx * self.h[c] + h, my * self.v[c] + v)))
                out.append(blocks)
        return out


def _kind(frame: _Frame, ss: int, ah: int) -> str:
    if not frame.progressive:
        return "seq"
    if ss == 0:
        return "dc_refine" if ah else "dc_first"
    return "ac_refine" if ah else "ac_first"


def _decode_interval(coef, bits: _Bits, mcus, kind, ss, se, al, dc_tabs, ac_tabs, cov, run_bits):
    """One restart interval (predictors and EOBRUN start at 0, T.81 F.2.1.3 / G.1.2.2)."""
    if kind == "seq":                                # DC and AC codes of sequential scans recorded apart
        lengths = cov["code_lengths"].setdefault("seq_dc", set())
        ac_lengths = cov["code_lengths"].setdefault("seq_ac", set())
    else:
        lengths = cov["code_lengths"].setdefault(kind, set())
    pred = [0, 0, 0]
    eobrun = 0
    p1, m1 = 1 << al, -1 << al
    for blocks in mcus:
        for k, row in blocks:
            blk = coef[row]
            if kind == "seq":                                            # F.2.2.1, F.2.2.2
                t = bits.decode(dc_tabs[k], lengths)
                pred[k] += _extend(bits.get(t), t)
                blk[0] = pred[k]
                i = 1
                while i < 64:
                    rs = bits.decode(ac_tabs[k], ac_lengths)
                    r, s = rs >> 4, rs & 15
                    if s:
                        i += r
                        if i > 63:
                            raise T81Error("coefficient past 63")
                        blk[i] = _extend(bits.get(s), s)
                        cov["seq_ac_nonzero"] += 1
                        i += 1
                    elif r == 15:
                        cov["seq_zrl"] += 1
                        i += 16
                    else:
                        break
            elif kind == "dc_first":                                     # G.1.2.1
                t = bits.decode(dc_tabs[k], lengths)
                pred[k] += _extend(bits.get(t), t)
                blk[0] = pred[k] * p1
            elif kind == "dc_refine":
                if bits.get(1):
                    blk[0] |= p1
            elif kind == "ac_first":                                     # G.1.2.2
                if eobrun:
                    eobrun -= 1
                    continue
                i = ss
                while i <= se:
                    rs = bits.decode(ac_tabs[0], lengths)
                    r, s = rs >> 4, rs & 15
                    if s:
                        i += r
                        if i > se:
                            raise T81Error("coefficient past Se")
                        blk[i] = _extend(bits.get(s), s) * p1
                    elif r == 15:
                        i += 15
                    else:
                        cov["eobn"]["ac_first"].add(r)
                        eobrun = (1 << r) + bits.get(r) - 1
                        break
                    i += 1
            else:                                                        # ac_refine, G.1.2.3
                i = ss
                if eobrun == 0:
                    while i <= se:
                        rs = bits.decode(ac_tabs[0], lengths)
                        r, s = rs >> 4, rs & 15
                        new = 0
                        if s:
                            if s != 1:
                                raise T81Error("refinement symbol of size other than 1")
                            new = p1 if bits.get(1) else m1
                        elif r != 15:
                            cov["eobn"]["ac_refine"].add(r)
                            eobrun = (1 << r) + bits.get(r)
                            run_bits[0] = 0
                            break
                        while i <= se:                                   # skip r zero coefficients, correcting the rest
                            c = int(blk[i])
                            if c:
                                if bits.get(1) and (c & p1) == 0:
                                    blk[i] = c + p1 if c >= 0 else c + m1
                            else:
                                if r == 0:
                                    break
                                r -= 1
                            i += 1
                        if new:
                            if i > se:
                                raise T81Error("new coefficient past Se")
                            blk[i] = new
                        i += 1
                if eobrun:                                               # inside an EOB run: correction bits only
                    for q in (i + np.flatnonzero(blk[i:se + 1])).tolist():
                        c = int(blk[q])
                        run_bits[0] += 1
                        if bits.get(1) and (c & p1) == 0:
                            blk[q] = c + p1 if c >= 0 else c + m1
                    eobrun -= 1
                    if eobrun == 0:
                        cov["max_eob_corrections"] = max(cov["max_eob_corrections"], run_bits[0])
    if run_bits[0]:
        cov["max_eob_corrections"] = max(cov["max_eob_corrections"], run_bits[0])
    run_bits[0] = 0


def decode(buf: bytes):
    """(coef int16 [blocks, 64], geometry dict, coverage dict) of a JPEG file; raises T81Error on what it cannot
    decode.  A file that ends early keeps the scans it has."""
    if buf[:2] != b"\xff\xd8":
        raise T81Error("no SOI")
    cov = dict(code_lengths={}, eobn={"ac_first": set(), "ac_refine": set()}, max_eob_corrections=0, fill_bytes=0,
               seq_ac_nonzero=0, seq_zrl=0, scan_comps=[], al={}, levels=0)
    tables = {}
    dri = 0
    frame = None
    coef = None
    level_of = {}                              # (component, coefficient) -> chain length of the last scan coding it
    i = 2
    while i + 1 < len(buf):
        if buf[i] != 0xFF:
            raise T81Error(f"marker expected at {i}")
        j = i + 1
        while j < len(buf) and buf[j] == 0xFF:
            j += 1
        cov["fill_bytes"] += j - i - 1
        if j >= len(buf):
            break
        m = buf[j]
        i = j + 1
        if m == 0xD9:
            break
        if 0xD0 <= m <= 0xD7 or m == 0x01:
            continue
        if i + 2 > len(buf):
            break
        ln = struct.unpack(">H", buf[i:i + 2])[0]
        p = buf[i + 2:i + ln]
        i += ln
        if m in (0xC0, 0xC1, 0xC2):
            frame = _Frame(p, m == 0xC2)
            coef = np.zeros((frame.mcus_x * frame.mcus_y * frame.bpm, 64), dtype=np.int64)
        elif m in (0xC3, 0xC5, 0xC6, 0xC7, 0xC9, 0xCA, 0xCB, 0xCD, 0xCE, 0xCF):
            raise T81Error("not a Huffman DCT frame")
        elif m == 0xC4:                                                  # B.2.4.2, any number of tables
            k = 0
            while k < len(p):
                tc, th = p[k] >> 4, p[k] & 15
                bits = list(p[k + 1:k + 17])
                n = sum(bits)
                tables[(tc, th)] = _huff(bits, p[k + 17:k + 17 + n])
                k += 17 + n
        elif m == 0xDD:
            dri = struct.unpack(">H", p[:2])[0]
        elif m == 0xDA:
            if frame is None:
                raise T81Error("scan before the frame")
            ns = p[0]
            comps, dc_tabs, ac_tabs = [], [], []
            for k in range(ns):
                comps.append(frame.ids.index(p[1 + 2 * k]))
                t = p[2 + 2 * k]
                dc_tabs.append(tables.get((0, t >> 4)))
                ac_tabs.append(tables.get((1, t & 15)))
            ss, se, ahal = p[1 + 2 * ns], p[2 + 2 * ns], p[3 + 2 * ns]
            ah, al = ahal >> 4, ahal & 15
            kind = _kind(frame, ss, ah)
            cov["scan_comps"].append(tuple(comps))
            cov["al"].setdefault(kind, set()).add(al)
            positions = [(c, q) for c in comps for q in range(ss, se + 1)]
            lv = 1 + max([level_of.get(x, 0) for x in positions], default=0)
            for x in positions:
                level_of[x] = lv
            cov["levels"] = max(cov["levels"], lv)
            intervals, i = _segment(buf, i, cov)
            mcus = frame.scan_mcus(comps)
            per = dri if dri else len(mcus)
            run_bits = [0]
            for n in range(-(-len(mcus) // per) if mcus else 0):
                data, rst = intervals[n] if n < len(intervals) else (b"", None)
                if n and rst is not None and rst != (n - 1) & 7:
                    raise T81Error(f"RST{rst} where RST{(n - 1) & 7} belongs")
                _decode_interval(coef, _Bits(data), mcus[n * per:(n + 1) * per], kind, ss, se, al, dc_tabs, ac_tabs,
                                 cov, run_bits)
    if frame is None:
        raise T81Error("no frame")
    geometry = dict(width=frame.width, height=frame.height, ncomp=frame.ncomp, hf=frame.h[0], vf=frame.v[0],
                    mcus_x=frame.mcus_x, mcus_y=frame.mcus_y)
    return coef.astype(np.int16), geometry, cov
