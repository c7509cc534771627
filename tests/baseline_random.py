"""Random baseline (SOF0 / SOF1) files for the two entropy kernels of single-scan files (kernel 1a for files with
restart intervals, kernel 1b for restart-free ones), and a stream that never self-synchronises.

random_case() draws coefficients (multiscan_random.random_coefficients plus ZRL chains that end in EOB, blocks with
all 63 AC coefficients and no EOB, magnitudes 2^s - 1 whose extra bits are all ones, and an optional DC walk that
wraps int16), Huffman tables per (class, id) of four kinds (multiscan_writer's "flat", "long", "mixed", and a table
with a single code), random table selectors per component (SOF1 when an id above 1 is used), a restart layout and
0xFF fill bytes before every RSTn and before EOI.  Its twin holds the same coefficients and quantisation tables,
written with the template's standard tables, the same restart interval and no fill: what the oracle decodes to the
expected RGB.

nonsync_case() builds a 4:4:4 stream in which every 1024-bit sub-sequence from the second on starts a block at a
block-in-MCU index other than 0, with all three components on the same two tables: a decoder that is wrong only
about the block's place in the MCU consumes exactly the same bits and never notices, so the speculative entry
states of kernel 1b form one chain of wrong states that only the synchronisation rounds can walk.  spec_states()
restates the speculative pass's entry rule in Python.

TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import numpy as np

from tests import jpeg_writer as jw
from tests import multiscan_random as mr
from tests import multiscan_writer as mw

SAMPLINGS = mr.SAMPLINGS
DC_SYMBOLS = list(range(12))
AC_SYMBOLS = [0x00, 0xF0] + [(r << 4) | s for r in range(16) for s in range(1, 11)]
KINDS = ("flat", "long", "mixed")
SUB_BITS = 1024                     # kernel 1b's sub-sequence: 128 de-stuffed bytes


# restart layouts: none, a DRI segment of 0, 1, MCUs - 1, MCUs, MCUs + 5, 65535 and a few small intervals
DRIS = [0, "dri0", 1, "m-1", "m", "m+5", 65535, 2, 3, 7]
# sizes from 1x1 to a few hundred pixels; MCU counts that are not multiples of 32 or 128
SIZES = [(1, 1), (17, 9), (37, 53), (61, 35), (64, 48), (120, 88), (333, 217), (8, 8), (255, 129), (200, 152)]
N_BATCH = 64


def batch_params(i: int) -> dict:
    """Keyword arguments of random_case for case i of the mixed batch: every sampling, size and restart layout,
    a forced int16 DC walk in every fifth case (restart-free, at least 64x48), shared tables in every ninth."""
    sampling = SAMPLINGS[i % len(SAMPLINGS)]
    w, h = SIZES[(3 * i + i // len(SIZES)) % len(SIZES)]
    dri = DRIS[(i // len(SAMPLINGS) + i) % len(DRIS)]
    wrap = None
    if i % 5 == i // 5 % 5:
        w, h, dri, wrap = max(w, 64), max(h, 48), 0, True
    return dict(seed=5000 + i, width=w, height=h, sampling=sampling, dri=dri, wrap=wrap,
                share=True if i % 9 == 4 else None)


def wrap16(v):
    return ((np.asarray(v, dtype=np.int64) + 0x8000) & 0xFFFF) - 0x8000


def _layout(geometry):
    """(blocks per MCU, component of each block of an MCU)."""
    ncomp = geometry["ncomp"]
    ny = geometry["hf"] * geometry["vf"] if ncomp == 3 else 1
    bpm = ny + 2 if ncomp == 3 else 1
    return bpm, [0 if b < ny else b - ny + 1 for b in range(bpm)]


def _extra_blocks(rng, coef, geometry, dri, wrap_comps, flat_comp):
    """Overwrites some blocks of `coef` (int64) with the kinds the catalogue of random_coefficients lacks; returns
    (the blocks whose trailing zeros are written as ZRLs before the EOB, whether a DC walk passed 32767)."""
    n = coef.shape[0]
    bpm, comp_of = _layout(geometry)
    zrl = set()
    for b in range(n):
        r = rng.random()
        blk = coef[b]
        if r < 0.12:                                          # ZRL chain that ends in EOB
            last = int(rng.integers(1, 47))
            blk[1:] = 0
            blk[1:last + 1] = np.where(rng.random(last) < 0.3, rng.integers(-40, 41, last), 0)
            blk[last] = int(rng.integers(1, 1024)) * int(rng.choice([-1, 1]))
            zrl.add(b)
        elif r < 0.2:                                         # coefficient 63 nonzero: no EOB
            blk[1:] = np.where(rng.random(63) < 0.3, rng.integers(-200, 201, 63), 0)
            blk[63] = int(rng.integers(1, 1024)) * int(rng.choice([-1, 1]))
        elif r < 0.32:                                        # 2^s - 1: all-ones extra bits, long FF 00 runs
            s = int(rng.integers(1, 11))
            blk[1:] = np.where(rng.random(63) < 0.8, (1 << s) - 1, 0)
    comp = np.array(comp_of * (n // bpm))
    mcu = np.arange(n) // bpm
    wrapped = False
    for c in wrap_comps:                                      # DC climbs by 2000 per block of c and wraps int16
        rows = np.flatnonzero(comp == c)
        start = (mcu[rows] % dri == 0) if dri else np.zeros(len(rows), bool)
        start[0] = True
        j = np.arange(len(rows)) - np.maximum.accumulate(np.where(start, np.arange(len(rows)), 0))
        coef[rows, 0] = wrap16(2000 * j)
        wrapped |= bool(np.any(2000 * j > 32767))
    if flat_comp is not None:                                 # one symbol per class: tables with a single code
        coef[comp == flat_comp] = 0
    return zrl, wrapped


def symbols(coef, geometry, dri, zrl_tail=(), dc_mod16=False):
    """Per component (DC categories, AC symbols) that jpeg_writer.rewrite codes for these blocks."""
    bpm, comp_of = _layout(geometry)
    out = [(set(), set()) for _ in range(geometry["ncomp"])]
    pred = [0, 0, 0]
    zrl_tail = set(zrl_tail)
    c64 = np.asarray(coef, dtype=np.int64)
    for b in range(c64.shape[0]):
        m, bi = divmod(b, bpm)
        if bi == 0 and dri and m % dri == 0:
            pred = [0, 0, 0]
        c = comp_of[bi]
        blk = c64[b]
        diff = int(blk[0]) - pred[c]
        if dc_mod16:
            diff = int(wrap16(diff))
        pred[c] = int(blk[0])
        out[c][0].add(abs(diff).bit_length())
        nz = np.flatnonzero(blk[1:]) + 1
        prev = 0
        for k in nz.tolist():
            run = k - prev - 1
            if run > 15:
                out[c][1].add(0xF0)
            out[c][1].add(((run % 16) << 4) | abs(int(blk[k])).bit_length())
            prev = k
        last = int(nz[-1]) if len(nz) else 0
        if b in zrl_tail and (62 - last) // 16:
            out[c][1].add(0xF0)
        if last < 63:
            out[c][1].add(0x00)
    return out


def single_table(symbol, rng):
    """(bits, vals): one code, of a random length 1..16 (all zeros, so never the all-ones code)."""
    bits = [0] * 16
    bits[int(rng.integers(0, 16))] = 1
    return bits, [symbol]


_POOL = {}


def shared_tables():
    """A DC and an AC table over the whole alphabet, the same content for every case that shares them."""
    if not _POOL:
        rng = np.random.default_rng(12345)
        _POOL["dc"] = mw.mixed_table(DC_SYMBOLS, rng)
        _POOL["ac"] = mw.mixed_table(AC_SYMBOLS, rng)
    return _POOL["dc"], _POOL["ac"]


def scan_range(f: bytes):
    """(first, end) byte offsets of the entropy-coded data of a single-scan file (end: the EOI's 0xFF, fill bytes
    included)."""
    _, at = jw.segments(f)
    end = len(f) - 2
    return at, end


def ff00_phases(f: bytes) -> set:
    """Offsets mod 16 of the FF of every stuffed FF 00 pair in the scan (files sit 16-byte aligned in the arena)."""
    a, e = scan_range(f)
    d = np.frombuffer(f, np.uint8)[a:e]
    i = np.flatnonzero((d[:-1] == 0xFF) & (d[1:] == 0x00))
    return set(((i + a) % 16).tolist())


def random_case(seed: int, width: int, height: int, sampling: str, dri=None, fill=None, wrap=None, share=None,
                port=None):
    """dict(file, twin, coef, geometry, tables, dri, fill, stats) of one random restart or restart-free baseline
    file.  dri: the restart interval, one of DRIS or a number (None: random among DRIS); fill: 0xFF bytes before each RSTn and EOI (None: random); wrap: the DC of
    some components climbs by 2000 per block and wraps int16 (None: random); share: use the shared tables of
    shared_tables() under random ids and DHT order (None: random).  coef is what the file codes, int16 with the DC
    wrapped to int16 as the reference decoder does."""
    rng = np.random.default_rng([seed, 77])
    tmpl = mr.template(width, height, sampling)
    g = port.decode(tmpl, entropy_only=True)["geometry"]
    ncomp = g["ncomp"]
    n_mcus = g["mcus_x"] * g["mcus_y"]
    if dri is None:
        dri = DRIS[int(rng.integers(len(DRIS)))]
    dri = {"m-1": n_mcus - 1, "m": n_mcus, "m+5": n_mcus + 5}.get(dri, dri)
    dri_segment = dri == "dri0"
    ri = 0 if dri_segment else max(0, min(65535, int(dri)))
    if fill is None:
        fill = int(rng.choice([0, 0, 0, 1, 2, 5]))
    if wrap is None:
        wrap = rng.random() < 0.3
    if share is None:
        share = rng.random() < 0.15
    flat_comp = None
    if not share and not wrap and rng.random() < 0.25:
        flat_comp = ncomp - 1 if ncomp == 3 else (0 if rng.random() < 0.4 else None)
    wrap_comps = [] if not wrap else ([0] if ncomp == 1 or rng.random() < 0.5 else list(range(ncomp)))

    coef = mr.random_coefficients(rng, g).astype(np.int64)
    zrl, wrapped = _extra_blocks(rng, coef, g, ri, wrap_comps, flat_comp)
    coef16 = coef.astype(np.int16)

    sof1 = flat_comp is not None or rng.random() < 0.5
    top = 4 if sof1 else 2
    if flat_comp is not None:                                 # its own ids, so its tables hold one symbol each
        sel = [(int(rng.integers(0, 3)), int(rng.integers(0, 3))) for _ in range(ncomp)]
        sel[flat_comp] = (3, 3)
    else:
        sel = [(int(rng.integers(0, top)), int(rng.integers(0, top))) for _ in range(ncomp)]
    need = symbols(coef16, g, ri, zrl, dc_mod16=True)
    tables, kinds = {}, {}
    for cls in (0, 1):
        for tid in sorted({s[cls] for s in sel}):
            if share:
                tables[(cls, tid)] = shared_tables()[cls]
                kinds[(cls, tid)] = "shared"
                continue
            syms = set().union(*[need[c][cls] for c in range(ncomp) if sel[c][cls] == tid])
            if len(syms) == 1 and rng.random() < 0.8:
                kinds[(cls, tid)] = "single"
                tables[(cls, tid)] = single_table(next(iter(syms)), rng)
                continue
            alphabet = DC_SYMBOLS if cls == 0 else AC_SYMBOLS
            extra = rng.choice(alphabet, int(rng.integers(0, 6)))
            kind = KINDS[int(rng.integers(3))]
            kinds[(cls, tid)] = kind
            tables[(cls, tid)] = mw.TABLES[kind](sorted(syms | set(int(x) for x in extra)), rng)
    order = list(tables)
    rng.shuffle(order)
    order = [tuple(int(v) for v in k) for k in order]
    decoy = None
    if rng.random() < 0.3:                                    # an id defined twice: the later DHT counts
        k = order[int(rng.integers(len(order)))]
        decoy = {k: ([1] + [0] * 15, [0x00 if k[0] else 0])}
    quant = {0: rng.integers(1, 17, 64), 1: rng.integers(1, 17, 64)}
    quant = quant if ncomp == 3 else {0: quant[0]}
    tq = [0, 1, 1][:ncomp]
    f = jw.blocks_to_jpeg(tmpl, coef16, g, quant, tq=tq, tables=tables, restart_interval=ri, selectors=sel,
                          fill=fill, dc_mod16=True, decoy=decoy, dht_order=order,
                          sof_marker=0xC1 if sof1 else 0xC0, dri_segment=dri_segment, zrl_tail=zrl)
    twin = jw.blocks_to_jpeg(tmpl, coef16, g, quant, tq=tq, restart_interval=ri, dc_mod16=True)
    longest_dc = max((L for (cls, _), (bits, _) in tables.items() if cls == 0 for L in range(1, 17) if bits[L - 1]))
    n_intervals = -(-n_mcus // ri) if ri else 1
    stats = dict(kinds=kinds, selectors=sel, sof1=sof1, wrap_comps=wrap_comps, flat_comp=flat_comp, share=share,
                 decoy=decoy is not None, zrl_blocks=len(zrl), dc16=longest_dc == 16, ff00=ff00_phases(f),
                 n_mcus=n_mcus, n_intervals=n_intervals, fill_before_rst=fill > 0 and n_intervals > 1,
                 dri_segment=dri_segment, wrapped=wrapped)
    return dict(file=f, twin=twin, coef=coef16, geometry=g, tables=tables, dri=dri, fill=fill, stats=stats)


# ---- a stream that never self-synchronises ---------------------------------------------------------------------
# DC: one 7-bit code (0000000) for category 1, so a DC symbol is that code and one bit: byte 00 (-1) or 01 (+1).
# AC: a 7-bit code (0000000) for 0x01 and an 8-bit one (00000010) for EOB: bytes 00 / 01 and 02.
NONSYNC_DC = ([0, 0, 0, 0, 0, 0, 1] + [0] * 9, [1])
NONSYNC_AC = ([0, 0, 0, 0, 0, 0, 1, 1] + [0] * 8, [0x01, 0x00])
# +-1 DC differences, a different pattern per component: a block decoded as the wrong component changes the slab
DC_PATTERNS = ([1, -1], [1, 1, -1, -1], [1, 1, 1, -1, -1, -1])


def nonsync_lengths(n_blocks: int, block_bytes: int | None = None) -> np.ndarray:
    """Bytes of each block.  Default: 64 blocks of 2 bytes in the first 128-byte sub-sequence, then per sub-sequence
    62 of 2 bytes and one of 4 (63 blocks: the block-in-MCU index at every boundary stays 64 mod 3 = 1).  With
    block_bytes: every block that long (3: the blocks do not divide 1024 bits)."""
    if block_bytes is not None:
        return np.full(n_blocks, block_bytes, np.int64)
    out = np.full(n_blocks, 2, np.int64)
    long_ = 64 + 31 + 63 * np.arange(max(0, (n_blocks - 64 + 62) // 63))
    out[long_[long_ < n_blocks]] = 4
    return out


def nonsync_case(width: int, height: int, block_bytes: int | None = None, port=None):
    """dict(file, coef, geometry, lengths) of a 4:4:4 restart-free file built byte by byte (no FF byte, so no
    stuffing: the de-stuffed stream is the scan itself)."""
    tmpl = mr.template(width, height, "4:4:4")
    g = port.decode(tmpl, entropy_only=True)["geometry"]
    n = g["mcus_x"] * g["mcus_y"] * 3
    lengths = nonsync_lengths(n, block_bytes)
    comp = np.arange(n) % 3
    diff = np.zeros(n, np.int64)
    for c in range(3):
        rows = np.flatnonzero(comp == c)
        pat = np.array(DC_PATTERNS[c])
        diff[rows] = pat[np.arange(len(rows)) % len(pat)]
    coef = np.zeros((n, 64), np.int64)
    for c in range(3):
        rows = np.flatnonzero(comp == c)
        coef[rows, 0] = np.cumsum(diff[rows])
    # block bytes: DC (00 / 01), then (len - 2) AC bytes of +-1, then EOB (02)
    ends = np.cumsum(lengths)
    starts = ends - lengths
    scan = np.full(int(ends[-1]), 0x02, np.uint8)
    scan[starts] = (diff > 0).astype(np.uint8)
    for extra in range(1, int(lengths.max()) - 1):
        rows = np.flatnonzero(lengths - 2 >= extra)
        sign = (rows + extra) % 2                              # +1, -1, ... along the block
        scan[starts[rows] + extra] = sign
        coef[rows, extra] = np.where(sign == 1, 1, -1)
    segs, _ = jw.segments(tmpl)
    out = bytearray(b"\xff\xd8")
    for m, p in segs:
        if m in (0xC4, 0xDA, 0xDD):
            continue
        out += jw._seg(m, p)
    out += jw._seg(0xC4, jw._dht_payload(0, 0, *NONSYNC_DC) + jw._dht_payload(1, 0, *NONSYNC_AC))
    sof = [p for m, p in segs if m == 0xC0][0]
    ids = [sof[6 + 3 * c] for c in range(3)]
    out += jw._seg(0xDA, bytes([3]) + b"".join(bytes([i, 0x00]) for i in ids) + bytes([0, 63, 0]))
    out += scan.tobytes() + b"\xff\xd9"
    return dict(file=bytes(out), coef=coef.astype(np.int16), geometry=g, lengths=lengths)


def _lookup(bits, vals):
    """16-bit window -> (code length, symbol), (0, None) where no code matches."""
    lut = [(0, None)] * 65536
    code, k = 0, 0
    for L in range(1, 17):
        for _ in range(bits[L - 1]):
            lo = code << (16 - L)
            for w in range(lo, lo + (1 << (16 - L))):
                lut[w] = (L, vals[k])
            code += 1
            k += 1
        code <<= 1
    return lut


def spec_decode(data: bytes, state, end_bit: int, dc_lut, ac_lut, bpm: int):
    """Kernel 1b's sub-sequence decoder restated: from state (bit, k, c) decode symbols, the same tables for every
    component, until the bit position reaches end_bit; returns the exit state.  (An undecodable code consumes one
    bit and ends the block; D has none.)"""
    p, k, c = state
    d = data + b"\x00" * 8
    while p < end_bit:
        w = (int.from_bytes(d[p >> 3:(p >> 3) + 4], "big") >> (16 - (p & 7))) & 0xFFFF
        L, sym = (ac_lut if k else dc_lut)[w]
        if L == 0:
            p, k = p + 1, 64
        elif k == 0:
            p, k = p + L + sym, 1
        else:
            r, s = sym >> 4, sym & 15
            p += L + s
            k = 64 if (s == 0 and r != 15) else k + r + 1
        if k >= 64:
            k, c = 0, (c + 1) % bpm
    return p, k, c


def spec_states(data: bytes, bpm: int = 3, dc=NONSYNC_DC, ac=NONSYNC_AC):
    """(x, e) per sub-sequence li of the speculative pass: x[li] is the exit state of decoding sub-sequence li - 1
    from (bit (li - 1) * 1024, k = 0, block 0) (x[0] the true start), e[li] the exit state of decoding sub-sequence
    li from x[li]."""
    dc_lut, ac_lut = _lookup(*dc), _lookup(*ac)
    n = -(-len(data) * 8 // SUB_BITS)
    x, e = [], []
    for li in range(n):
        xs = (0, 0, 0) if li == 0 else spec_decode(data, ((li - 1) * SUB_BITS, 0, 0), li * SUB_BITS, dc_lut, ac_lut, bpm)
        x.append(xs)
        e.append(spec_decode(data, xs, (li + 1) * SUB_BITS, dc_lut, ac_lut, bpm))
    return x, e


def true_states(lengths: np.ndarray, bpm: int = 3):
    """The state of a sequential decode at every sub-sequence boundary of a stream whose blocks start at every
    boundary (D's layout): (bit, 0, block-in-MCU of the block that starts there)."""
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]) * 8
    n = -(-int(np.sum(lengths)) * 8 // SUB_BITS)
    idx = np.searchsorted(starts, np.arange(n) * SUB_BITS)
    return [(li * SUB_BITS, 0, int(idx[li]) % bpm) if idx[li] < len(starts) and starts[idx[li]] == li * SUB_BITS
            else None for li in range(n)]

