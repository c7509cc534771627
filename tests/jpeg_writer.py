"""A small baseline-JPEG re-writer for tests: takes an existing baseline file, its entropy-decoded
coefficients (from the oracle) and re-emits the scan with other Huffman tables / restart intervals /
header oddities.  Used to hand-build inputs no encoder in this image writes: 16-bit DC codes
(loadjpg.cpp:562 cannot decode them), crafted DHTs, non-interleaved SOS headers, 12-bit SOF.

TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import struct

import numpy as np


def segments(jpg: bytes):
    """[(marker, payload)] of everything between SOI and the scan, and the offset of the scan data."""
    assert jpg[:2] == b"\xff\xd8"
    out, i = [], 2
    while True:
        assert jpg[i] == 0xFF, hex(jpg[i])
        m = jpg[i + 1]
        i += 2
        if m == 0xFF:
            i -= 1
            continue
        n = struct.unpack(">H", jpg[i:i + 2])[0]
        out.append((m, jpg[i + 2:i + n]))
        i += n
        if m == 0xDA:
            return out, i


def dht_tables(segs):
    """{(class, id): (bits[16], vals)} from the DHT segments."""
    t = {}
    for m, p in segs:
        if m != 0xC4:
            continue
        k = 0
        while k < len(p):
            tc, th = p[k] >> 4, p[k] & 15
            bits = list(p[k + 1:k + 17])
            n = sum(bits)
            t[(tc, th)] = (bits, list(p[k + 17:k + 17 + n]))
            k += 17 + n
    return t


def canonical_codes(bits, vals):
    """symbol -> (code, length), the assignment of GenHuffCodes (openjpg.cpp:48-66) / JPEG Annex C."""
    codes, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            codes[vals[k]] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return codes


class BitWriter:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, value: int, nbits: int):
        if nbits == 0:
            return
        self.acc = (self.acc << nbits) | (value & ((1 << nbits) - 1))
        self.n += nbits
        while self.n >= 8:
            b = (self.acc >> (self.n - 8)) & 0xFF
            self.out.append(b)
            if b == 0xFF:
                self.out.append(0)          # byte stuffing
            self.n -= 8
        self.acc &= (1 << self.n) - 1

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)     # pad with ones


def _seg(marker: int, payload: bytes) -> bytes:
    return bytes([0xFF, marker]) + struct.pack(">H", len(payload) + 2) + payload


def _dht_payload(tc, th, bits, vals) -> bytes:
    return bytes([(tc << 4) | th]) + bytes(bits) + bytes(vals)


def _dqt_payload(tid: int, q) -> bytes:
    q = [int(v) for v in q]
    assert len(q) == 64 and all(1 <= v <= 255 for v in q), "8-bit tables, zig-zag order"
    return bytes([tid]) + bytes(q)


def rewrite(jpg: bytes, coef: np.ndarray, geometry: dict, tables: dict | None = None, restart_interval: int = 0,
            sof_precision: int | None = None, sos_override: bytes | None = None, trailer: bytes = b"\xff\xd9",
            quant: dict | None = None, tq: list | None = None, selectors: list | None = None, fill: int = 0,
            dc_mod16: bool = False, decoy: dict | None = None, dht_order: list | None = None,
            sof_marker: int | None = None, dri_segment: bool = False, zrl_tail=()) -> bytes:
    """Re-emit `jpg` (baseline, decoded to `coef` [blocks, 64] zig-zag with absolute DC, scan order) with the
    Huffman tables of `tables` ({(class, id): (bits, vals)} overriding the file's own), a new restart interval,
    and optional header oddities.  `quant` ({table id: 64 values, zig-zag order}) replaces the file's DQT segments;
    `tq` sets each component's quantisation table selector in the SOF.
    selectors: per component (DC id, AC id), written to the SOS (default: the file's own SOS).
    fill: that many 0xFF fill bytes (T.81 B.1.1.2) before every RSTn and before the trailer.
    dc_mod16: DC differences taken modulo 2^16 (in [-32768, 32767]), so that an absolute DC sequence may wrap the
    int16 range of `coef` as a decoder that keeps its predictor in int16 does.
    decoy: {(class, id): (bits, vals)} written in a DHT before the real tables, which redefine every such id.
    dht_order: the (class, id) keys in the order their DHT segments are written (default: sorted).
    sof_marker: 0xC0 / 0xC1 for the frame header (default: the file's).  dri_segment: write a DRI segment even for
    restart_interval 0.  zrl_tail: blocks whose trailing zeros are coded as ZRLs before the EOB (as far as the
    ZRLs stay inside the block; T.81 allows it, libjpeg never writes it)."""
    segs, _ = segments(jpg)
    tabs = dht_tables(segs)
    if tables:
        tabs.update(tables)
    sof = [p for m, p in segs if m in (0xC0, 0xC1)][0]
    sos = [p for m, p in segs if m == 0xDA][0]
    ncomp = sof[5]
    comp_ids = [sof[6 + 3 * c] for c in range(ncomp)]
    if selectors is not None:
        sos = bytes([ncomp]) + b"".join(bytes([comp_ids[c], (selectors[c][0] << 4) | selectors[c][1]])
                                         for c in range(ncomp)) + sos[1 + 2 * sos[0]:]
    sel = {}
    for k in range(sos[0]):
        cs, t = sos[1 + 2 * k], sos[2 + 2 * k]
        sel[comp_ids.index(cs)] = (t >> 4, t & 15)
    zrl_tail = set(int(b) for b in zrl_tail)
    codes = {key: canonical_codes(*tabs[key]) for key in tabs}

    hf, vf = geometry["hf"], geometry["vf"]
    ny = hf * vf if ncomp == 3 else 1
    bpm = ny + 2 if ncomp == 3 else 1
    n_mcus = geometry["mcus_x"] * geometry["mcus_y"]
    assert coef.shape[0] == n_mcus * bpm

    bw = BitWriter()
    pred = [0, 0, 0]
    rst = 0
    scan = bytearray()
    for mcu in range(n_mcus):
        if restart_interval and mcu and mcu % restart_interval == 0:
            bw.flush()
            scan += bw.out + b"\xff" * fill + bytes([0xFF, 0xD0 + (rst & 7)])
            bw = BitWriter()
            pred = [0, 0, 0]
            rst += 1
        for bi in range(bpm):
            comp = 0 if bi < ny else bi - ny + 1
            dc_codes, ac_codes = codes[(0, sel[comp][0])], codes[(1, sel[comp][1])]
            blk = coef[mcu * bpm + bi].astype(np.int64)
            diff = int(blk[0]) - pred[comp]
            if dc_mod16:
                diff = ((diff + 0x8000) & 0xFFFF) - 0x8000
            pred[comp] = int(blk[0])
            cat = abs(diff).bit_length()
            if cat not in dc_codes:
                raise ValueError(f"DC difference {diff} (MCU {mcu}, block {bi}) has no code in the DC table")
            c, length = dc_codes[cat]
            bw.put(c, length)
            bw.put(diff if diff >= 0 else diff + (1 << cat) - 1, cat)
            run = 0
            last = int(np.max(np.nonzero(blk[1:])[0])) + 1 if np.any(blk[1:]) else 0
            for k in range(1, last + 1):
                v = int(blk[k])
                if v == 0:
                    run += 1
                    continue
                while run > 15:
                    c, length = ac_codes[0xF0]
                    bw.put(c, length)
                    run -= 16
                size = abs(v).bit_length()
                c, length = ac_codes[(run << 4) | size]
                bw.put(c, length)
                bw.put(v if v >= 0 else v + (1 << size) - 1, size)
                run = 0
            if mcu * bpm + bi in zrl_tail:
                for _ in range((62 - last) // 16):
                    c, length = ac_codes[0xF0]
                    bw.put(c, length)
            if last < 63:
                c, length = ac_codes[0x00]
                bw.put(c, length)
    bw.flush()
    scan += bw.out + b"\xff" * fill

    out = bytearray(b"\xff\xd8")
    dqt_done = False
    for m, p in segs:
        if m in (0xC4, 0xDA, 0xDD):
            continue
        if m == 0xDB and quant is not None:
            if not dqt_done:                    # all of `quant` where the file's first DQT was
                for tid, q in sorted(quant.items()):
                    out += _seg(0xDB, _dqt_payload(tid, q))
                dqt_done = True
            continue
        if m in (0xC0, 0xC1) and sof_precision is not None:
            p = bytes([sof_precision]) + p[1:]
        if m in (0xC0, 0xC1) and tq is not None:
            p = bytearray(p)
            for c in range(ncomp):
                p[6 + 3 * c + 2] = tq[c]
            p = bytes(p)
        if m in (0xC0, 0xC1) and sof_marker is not None:
            m = sof_marker
        out += _seg(m, p)
    if decoy:
        out += _seg(0xC4, b"".join(_dht_payload(tc, th, *decoy[(tc, th)]) for tc, th in sorted(decoy)))
    for tc, th in (sorted(tabs) if dht_order is None else dht_order):
        out += _seg(0xC4, _dht_payload(tc, th, *tabs[(tc, th)]))
    if restart_interval or dri_segment:
        out += _seg(0xDD, struct.pack(">H", restart_interval))
    out += _seg(0xDA, sos_override if sos_override is not None else sos)
    out += scan + trailer
    return bytes(out)


def block_index(geometry: dict, ncomp: int, mcu: int, comp: int, sub: int = 0) -> int:
    """Row of the [blocks, 64] scan-order coefficient array that holds block `sub` (luma: raster order inside the MCU)
    of component `comp` in MCU `mcu`."""
    ny = geometry["hf"] * geometry["vf"] if ncomp == 3 else 1
    bpm = ny + 2 if ncomp == 3 else 1
    assert (sub < ny) if comp == 0 else sub == 0
    return mcu * bpm + (sub if comp == 0 else ny + comp - 1)


def blocks_to_jpeg(template: bytes, blocks: np.ndarray, geometry: dict, quant: dict, tq: list | None = None,
                   tables: dict | None = None, restart_interval: int = 0, **kw) -> bytes:
    """A baseline file that holds exactly `blocks` ([blocks, 64] int, zig-zag order, absolute DC, MCU / scan order).
    `template` gives size, sampling and Huffman tables: a file written by PIL with its standard tables, which code
    every DC category 0-11 and every AC run/size; `geometry` is its port.decode(..., entropy_only=True)["geometry"].
    `quant` ({id: 64 values, zig-zag}) and `tq` (table id per component, default 0, 1, 1 / 0) are the
    quantisation tables written.  Further keyword arguments go to rewrite()."""
    ncomp = geometry["ncomp"]
    if tq is None:
        tq = [0, 1, 1][:ncomp]
    return rewrite(template, np.asarray(blocks), geometry, tables=tables, restart_interval=restart_interval,
                   quant=quant, tq=tq, **kw)


def replace_tables(jpg: bytes, tables: dict, sof_precision: int | None = None, sos_override: bytes | None = None) -> bytes:
    """Same file, same scan bytes, other DHT contents / SOF precision / SOS header: for crafted (hostile) inputs."""
    segs, scan_at = segments(jpg)
    tabs = dht_tables(segs)
    tabs.update(tables)
    out = bytearray(b"\xff\xd8")
    for m, p in segs:
        if m in (0xC4, 0xDA):
            continue
        if m in (0xC0, 0xC1) and sof_precision is not None:
            p = bytes([sof_precision]) + p[1:]
        out += _seg(m, p)
    for (tc, th), (bits, vals) in sorted(tabs.items()):
        out += _seg(0xC4, _dht_payload(tc, th, bits, vals))
    sos = [p for m, p in segs if m == 0xDA][0]
    out += _seg(0xDA, sos_override if sos_override is not None else sos)
    out += jpg[scan_at:]
    return bytes(out)


# A DC table whose category-2 symbol (differences of +-2..3, frequent in any image) has a 16-bit code:
# lengths 1..11 for categories 1, 0, 3, 4, ..., 11 (codes 0, 10, 110, ...), then 1111111111100000 for 2.
DC16_BITS = [1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 1]
DC16_VALS = [1, 0, 3, 4, 5, 6, 7, 8, 9, 10, 11, 2]

# An AC table in which every code is a size-0 symbol with a run other than 0 and 15: the reference ignores
# those (loadjpg.cpp:771-775) and so never reaches the end of a block (it spins forever, 700-829).
STUCK_AC_BITS = [1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2]
STUCK_AC_VALS = [0x10] * 17
