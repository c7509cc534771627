"""CPU tests of the product's host side: the C-ABI library builds, loads, exports every symbol
include/hjd.h declares, parses headers, writes BMPs, and refuses to decode without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from tests import cases


def declared_symbols(header_path):
    text = open(header_path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hjd_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(hjd):
    L = ctypes.CDLL(hjd.LIB_PATH)
    names = declared_symbols(hjd.INCLUDE_PATH)
    assert len(names) >= 35
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert hjd.lib().hjd_version() == 100


def test_reference_cxx_names_are_exported(hjd):
    """csrc/ref_shim.cpp: the reference's own (C++-mangled) entry points."""
    import subprocess
    out = subprocess.check_output(["nm", "-DC", hjd.LIB_PATH], text=True)
    assert "ConvertJpgFile(char*, char*)" in out
    assert "DecodeJpgFileData(unsigned char const*, int, unsigned char**, unsigned int*, unsigned int*)" in out
    assert "WriteBMP24(char const*, unsigned int, unsigned int, unsigned char*)" in out


def test_image_size_from_header(hjd):
    for name, jpg in cases.small_cases().items():
        w, h = hjd.JpegGetImageSize(jpg)
        m = re.search(r"_(\d+)x(\d+)", name)
        if m:
            assert (w, h) == (int(m.group(1)), int(m.group(2))), name
    with pytest.raises(hjd.HjdError):
        hjd.JpegGetImageSize(cases.progressive_jpeg())
    with pytest.raises(hjd.HjdError):
        hjd.JpegGetImageSize(b"\xff\xd8\xff")
    with pytest.raises(hjd.HjdError):
        hjd.JpegGetImageSize(cases.cmyk_jpeg())


def test_truncated_headers_never_crash(hjd):
    jpg = cases.small_cases()["420_100x70_ri2"]
    for cut in range(0, 700, 7):
        try:
            hjd.JpegGetImageSize(jpg[:cut])
        except hjd.HjdError:
            pass


def test_bmp_bytes_match_oracle(hjd, port, tmp_path):
    for (w, h) in [(1, 1), (2, 3), (13, 7), (16, 16), (5, 9)]:
        rgb = cases.noise_rgb(w, h, w * 100 + h)
        want = port.bmp24_bytes(rgb)
        assert hjd.encode_bmp24(rgb) == want
        p = str(tmp_path / f"o_{w}x{h}.bmp")
        hjd.WriteBMP24(p, w, h, rgb)
        assert open(p, "rb").read() == want
        assert len(want) == w * h * 3 + h * ((4 - (w * 3) % 4) % 4) + 54


def test_idct_constants_match_oracle(hjd, port):
    c, cc = hjd.idct_tables()
    oc, occ = port.idct_tables()
    assert np.array_equal(c, oc) and np.array_equal(cc, occ)
    assert (c[:, 0] == 1.0).all()          # the kernels rely on cos(0) == 1 exactly


def test_no_gpu_means_loud_failure(hjd, tmp_path):
    if hjd.lib().hjd_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(hjd.HjdError, match="no CUDA device"):
        hjd.BatchDecoder(0)
    with pytest.raises(hjd.HjdError):
        hjd.DecodeJpgFileData(cases.small_cases()["444_1x1"])
    assert hjd.ConvertJpgFile(str(tmp_path / "missing.jpg"), str(tmp_path / "x.bmp")) == 0


def test_product_does_not_touch_the_oracle():
    """The shipped package must not import, include, link or execute anything under oracle/."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "hls_jpeg_decoder_b200")
    bad = re.compile(r"^\s*(from|import)\s+oracle\b|#\s*include[^\n]*oracle|liboracle|jpeg_oracle|hjdo_|hjdref_|CDLL\([^)]*oracle",
                     re.M)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert not bad.search(text), (dirpath, f, bad.search(text).group(0))


# ---------------------------------------------------------------------------------------------
# round 2: two-level Huffman tables, probe, inputs beyond the reference (SURVEY.md 8(f) rank 4)
# ---------------------------------------------------------------------------------------------
def _std_tables():
    from tests import jpeg_writer as jw
    segs, _ = jw.segments(cases.small_cases()["420_64x48_q85"])
    return jw.dht_tables(segs)


def _brute_lookup(bits, vals, peek16):
    """(length, symbol) of the canonical code that prefixes the 16 bits, or None (openjpg.cpp:48-66 codes)."""
    code, k = 0, 0
    for length in range(1, 17):
        n = bits[length - 1]
        top = peek16 >> (16 - length)
        if code <= top < code + n:
            return length, vals[k + (top - code)]
        code = (code + n) << 1
        k += n
    return None


def _fields(length, sym, is_ac):
    size, run = sym & 15, sym >> 4
    if not is_ac:
        return length | size << 5 | 1 << 9
    if size:
        return length | size << 5 | (run + 1) << 9
    return length | (63 if run == 0 else 16 if run == 15 else 0) << 9


def test_two_level_huffman_tables_match_the_canonical_code_walk(hjd):
    """The kernels' lookup (10-bit first level + sub-tables for longer codes), built by the host from BITS /
    HUFFVAL, against the canonical code walk, for every possible 16-bit window: the standard tables, the
    16-bit-DC-code table, a full 16-bit-deep table and random (also incomplete) ones."""
    import ctypes as C
    from tests import jpeg_writer as jw
    L = hjd.lib()
    rng = np.random.default_rng(11)
    tables = [(b, v, tc) for (tc, _), (b, v) in _std_tables().items()]
    tables.append((jw.DC16_BITS, jw.DC16_VALS, 0))
    tables.append((jw.STUCK_AC_BITS, jw.STUCK_AC_VALS, 1))
    for _ in range(6):                           # random prefix codes: split the code space at random depths
        bits, space = [0] * 16, 1.0
        for length in range(1, 17):
            cap = int(space * (1 << length) + 1e-9)
            n = int(rng.integers(0, min(cap, 12 if length < 16 else 40) + 1)) if length > 1 else int(rng.integers(0, 2))
            n = min(n, 256 - sum(bits))
            bits[length - 1] = n
            space -= n / (1 << length)
        vals = [int(x) for x in rng.integers(0, 256, size=sum(bits))]
        tables.append((bits, vals, int(rng.integers(0, 2))))
    step = 1
    for bits, vals, is_ac in tables:
        bb = (C.c_uint8 * 16)(*bits)
        vv = (C.c_uint8 * max(len(vals), 1))(*vals)
        for peek in range(0, 65536, step):
            got = L.hjd_huff_lookup_probe(bb, vv, len(vals), is_ac, peek)
            want = _brute_lookup(bits, vals, peek)
            if want is None:
                assert got == 0xFE01, (bits, peek, got)          # HJD_BAD_ENTRY: one bit, advance 127
            else:
                assert got == _fields(want[0], want[1], bool(is_ac)), (bits, hex(peek), want, got)
    over = [2, 1] + [0] * 14                     # three codes in a 2-bit space cannot exist
    assert L.hjd_huff_lookup_probe((C.c_uint8 * 16)(*over), (C.c_uint8 * 3)(1, 2, 3), 3, 0, 0) == 0xFFFFFFFF


def test_probe_reports_what_a_batch_would(hjd):
    """hjd_probe_jpeg: geometry of decodable files; explicit rejection (HJD_IMG_ERR_UNSUPPORTED = -3) of
    12-bit precision, non-interleaved scans, progressive and CMYK files -- none of which the reference can
    decode either (SURVEY.md 8a footnote)."""
    from tests import jpeg_writer as jw
    base = cases.small_cases()
    st, inf = hjd.probe(base["420_100x70_ri2"])
    assert st == 0 and (inf.width, inf.height, inf.hf, inf.vf, inf.restart_interval) == (100, 70, 2, 2, 2)
    assert inf.n_blocks == 7 * 5 * 6 and inf.n_intervals == 18
    twelve = jw.replace_tables(base["444_64x48_q85"], {}, sof_precision=12)
    assert hjd.probe(twelve)[0] == -3
    one_component_scan = jw.replace_tables(base["444_64x48_q85"], {}, sos_override=bytes([1, 1, 0x00, 0, 63, 0]))
    assert hjd.probe(one_component_scan)[0] == -3
    assert hjd.probe(cases.progressive_jpeg())[0] == -3
    assert hjd.probe(cases.cmyk_jpeg())[0] == -3
    assert hjd.probe(b"")[0] == -1 and hjd.probe(b"\xff\xd8\xff")[0] == -1 and hjd.probe(b"\xff\xd8\xff\xe0\x00")[0] == -2
    over = jw.replace_tables(base["444_64x48_q85"], {(0, 0): ([2, 1] + [0] * 14, [0, 1, 2])})
    assert hjd.probe(over)[0] == -4              # HJD_IMG_ERR_BAD_TABLE


def test_scan_ends_at_the_first_real_marker(hjd):
    """ADVICE r1: what follows EOI (padding, a second image, a caller's oversized buffer) is not entropy data."""
    jpg = cases.small_cases()["420_100x70_ri2"]
    n0 = hjd.probe(jpg)[1].scan_bytes
    assert n0 == len(jpg) - jpg.rfind(b"\xff\xda") - 14 - 2     # SOS header is 2 + 12 bytes; EOI excluded
    trailer = jpg + b"\x00" * 1000 + b"\xff\xd3\xff\xd4" + jpg
    assert hjd.probe(trailer)[1].scan_bytes == n0
    assert hjd.probe(jpg[:-2])[1].scan_bytes == n0              # EOI missing: everything up to the end


def test_dc16_writer_and_oracle_switch(port):
    """A file whose DC table has a 16-bit code (tests/jpeg_writer.py): the reference's k = 1..15 search
    (loadjpg.cpp:562) cannot decode it; with the oracle's documented deviation switch it yields the
    coefficients of the source file."""
    from tests import jpeg_writer as jw
    src = cases.small_cases()["420_100x70_ri2"]
    o = port.decode(src, entropy_only=True)
    f = jw.rewrite(src, o["coef"], o["geometry"], tables={(0, 0): (jw.DC16_BITS, jw.DC16_VALS)}, restart_interval=2)
    try:
        port.set_dc16(True)
        o16 = port.decode(f, entropy_only=True)
        assert o16["rc"] == 0 and np.array_equal(o16["coef"], o["coef"])
    finally:
        port.set_dc16(False)
    o15 = port.decode(f, entropy_only=True)
    assert o15["rc"] != 0 or not np.array_equal(o15["coef"], o["coef"])     # the reference deviates here
    # the writer itself: same tables, other restart interval -> same coefficients
    g = jw.rewrite(src, o["coef"], o["geometry"], restart_interval=5)
    assert np.array_equal(port.decode(g, entropy_only=True)["coef"], o["coef"])
