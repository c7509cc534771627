"""Hand-built Exif APP1 segments, spliced after the SOI of an existing JPEG (which changes no coefficient).

tiff() writes the TIFF structure of an Exif payload in either byte order: IFD0 with optional entries before and after
the orientation tag 0x0112, and optionally an ExifIFD (tag 0x8769) and an IFD1 (the thumbnail's IFD, chained from IFD0),
each of which can carry an orientation of its own.  Fields can be set wrong on purpose (type, count, value, offsets)."""
from __future__ import annotations

import struct

SHORT, LONG = 3, 4
# (tag, type, count, value) of unrelated IFD0 entries, in tag order around 0x0112
BEFORE = [(0x0100, LONG, 1, 640), (0x0101, LONG, 1, 480)]
AFTER = [(0x0128, SHORT, 1, 2), (0x0213, SHORT, 1, 1)]


def _entry(order: str, tag: int, typ: int, count: int, value: int) -> bytes:
    val = struct.pack(order + "HH", value & 0xFFFF, 0) if typ == SHORT else struct.pack(order + "I", value & 0xFFFFFFFF)
    return struct.pack(order + "HHI", tag, typ, count) + val


def _ifd(order: str, entries, next_off: int = 0) -> bytes:
    return (struct.pack(order + "H", len(entries)) + b"".join(_entry(order, *e) for e in entries)
            + struct.pack(order + "I", next_off))


def tiff(orientation: int | None, order: str = "<", before=(), after=(), typ: int = SHORT, count: int = 1,
         exif_ifd_orientation: int | None = None, ifd1_orientation: int | None = None, ifd0_offset: int = 8,
         entry_count: int | None = None) -> bytes:
    """The TIFF structure.  orientation None: IFD0 has no 0x0112 entry.  entry_count: IFD0's count field as written
    (default: the true count)."""
    mark = b"II*\x00" if order == "<" else b"MM\x00*"
    entries = list(before)
    if orientation is not None:
        entries.append((0x0112, typ, count, orientation))
    entries += list(after)
    n0 = len(entries) + (exif_ifd_orientation is not None)
    ifd0_len = 2 + 12 * n0 + 4
    at = 8 + ifd0_len                                   # the sub-IFDs follow IFD0
    tail = b""
    if exif_ifd_orientation is not None:
        entries.append((0x8769, LONG, 1, at))
        sub = _ifd(order, [(0x0112, SHORT, 1, exif_ifd_orientation)])
        tail += sub
        at += len(sub)
    next_off = 0
    if ifd1_orientation is not None:
        next_off = at
        tail += _ifd(order, [(0x0112, SHORT, 1, ifd1_orientation)])
    body = _ifd(order, entries, next_off)
    if entry_count is not None:
        body = struct.pack(order + "H", entry_count) + body[2:]
    return mark + struct.pack(order + "I", ifd0_offset) + body + tail


def exif_payload(orientation: int | None, **kw) -> bytes:
    return b"Exif\x00\x00" + tiff(orientation, **kw)


def app1(payload: bytes) -> bytes:
    assert len(payload) + 2 <= 0xFFFF
    return b"\xff\xe1" + struct.pack(">H", len(payload) + 2) + payload


def xmp_app1() -> bytes:
    """An XMP APP1, which can carry an orientation too; it is not read."""
    return app1(b"http://ns.adobe.com/xap/1.0/\x00<x:xmpmeta><tiff:Orientation>6</tiff:Orientation></x:xmpmeta>")


def splice(jpg: bytes, *segments: bytes) -> bytes:
    """The file with `segments` inserted right after its SOI."""
    assert jpg[:2] == b"\xff\xd8"
    return jpg[:2] + b"".join(segments) + jpg[2:]


def with_orientation(jpg: bytes, orientation: int | None, **kw) -> bytes:
    return splice(jpg, app1(exif_payload(orientation, **kw)))


def after_sos(jpg: bytes, segment: bytes) -> bytes:
    """The file with `segment` inserted right before its EOI (after the scan), where no parser looks for Exif."""
    assert jpg[-2:] == b"\xff\xd9"
    return jpg[:-2] + segment + jpg[-2:]
