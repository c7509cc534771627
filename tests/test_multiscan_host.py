"""HJD_FLAG_MULTI_SCAN on the host (no GPU): the multi-scan parse behind probe(buf, FLAG_MULTI_SCAN) and scans(),
the T.81 G.1.1.1 checks, the scan cap, and the test writer (tests/multiscan_writer.py) against Pillow."""
from __future__ import annotations

import io
import struct

import numpy as np
import pytest
from PIL import Image

from tests import multiscan_writer as mw
from tests.cases import encode_jpeg_cv, small_cases
from tests.jpeg_writer import _seg
from tools.gen_jpegs import SUBSAMPLING, synth_rgb

GEOM = ["width", "height", "hf", "vf", "mcus_x", "mcus_y", "n_blocks"]


def pil_pair(rgb, sub="4:2:0", gray=False, restart=0, quality=85):
    """(progressive, baseline twin) written by libjpeg-turbo from the same pixels."""
    out = []
    for prog in (True, False):
        im = Image.fromarray(rgb)
        kw = dict(format="JPEG", quality=quality, progressive=prog)
        if gray:
            im = im.convert("L")
        else:
            kw["subsampling"] = SUBSAMPLING[sub]
        if restart:
            kw["restart_marker_blocks"] = restart
        buf = io.BytesIO()
        im.save(buf, **kw)
        out.append(buf.getvalue())
    return out


def cv_pair(rgb, sampling="440"):
    import cv2
    base = encode_jpeg_cv(rgb, 85, sampling)
    ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(rgb[:, :, ::-1]),
                           [cv2.IMWRITE_JPEG_QUALITY, 85, cv2.IMWRITE_JPEG_PROGRESSIVE, 1,
                            cv2.IMWRITE_JPEG_SAMPLING_FACTOR, getattr(cv2, "IMWRITE_JPEG_SAMPLING_FACTOR_" + sampling)])
    assert ok
    return buf.tobytes(), base


PAIRS = {
    "420_333x217": lambda: pil_pair(synth_rgb(333, 217, 1), "4:2:0"),
    "422_333x217": lambda: pil_pair(synth_rgb(333, 217, 2), "4:2:2"),
    "444_333x217": lambda: pil_pair(synth_rgb(333, 217, 3), "4:4:4"),
    "440_cv_61x35": lambda: cv_pair(synth_rgb(61, 35, 4), "440"),
    "gray_33x9": lambda: pil_pair(synth_rgb(33, 9, 5), gray=True),
    "420_1x1": lambda: pil_pair(synth_rgb(1, 1, 6), "4:2:0"),
    "444_1x1": lambda: pil_pair(synth_rgb(1, 1, 7), "4:4:4"),
    "420_37x53": lambda: pil_pair(synth_rgb(37, 53, 8), "4:2:0"),
    "420_100x70_ri2": lambda: pil_pair(synth_rgb(100, 70, 9), "4:2:0", restart=2),
    "444_48x40_ri1": lambda: pil_pair(synth_rgb(48, 40, 10), "4:4:4", restart=1),
}


@pytest.mark.parametrize("name", sorted(PAIRS))
def test_progressive_probe_matches_twin(hjd, name):
    prog, base = PAIRS[name]()
    st0, _ = hjd.probe(prog)
    assert st0 == -3                                            # without the flag: unsupported, as before
    st, o = hjd.probe(prog, hjd.FLAG_MULTI_SCAN)
    stb, ob = hjd.probe(base)
    assert st == 0 and stb == 0
    assert [getattr(o, k) for k in GEOM] == [getattr(ob, k) for k in GEOM]
    sc = hjd.scans(prog)
    assert o.scan_bytes == sum(s["bytes"] for s in sc)
    assert o.restart_interval == sc[0]["restart_interval"]
    assert hjd.scans(base) == [dict(ncomp=ob.ncomp, comp=list(range(ob.ncomp)), ss=0, se=63, ah=0, al=0, level=0,
                                    restart_interval=ob.restart_interval, bytes=ob.scan_bytes)]


def test_libjpeg_default_scripts(hjd):
    prog, _ = PAIRS["420_333x217"]()
    sc = hjd.scans(prog)
    assert [(tuple(s["comp"]), s["ss"], s["se"], s["ah"], s["al"]) for s in sc] == mw.DEFAULT_SCRIPT_COLOR
    assert [s["level"] for s in sc] == [0, 0, 0, 0, 0, 1, 1, 1, 1, 2]
    gray, _ = PAIRS["gray_33x9"]()
    sc = hjd.scans(gray)
    assert [(tuple(s["comp"]), s["ss"], s["se"], s["ah"], s["al"]) for s in sc] == mw.DEFAULT_SCRIPT_GRAY
    assert [s["level"] for s in sc] == [0, 0, 0, 1, 1, 2]


# A custom script: DC scans not interleaved, DC successive approximation, single-coefficient bands, Al up to 5.
CUSTOM_SCRIPT = [((0,), 0, 0, 0, 2), ((1,), 0, 0, 0, 1), ((2,), 0, 0, 0, 0), ((0,), 0, 0, 2, 1), ((0,), 0, 0, 1, 0),
                 ((1,), 0, 0, 1, 0), ((0,), 1, 1, 0, 5), ((0,), 2, 63, 0, 3), ((0,), 1, 1, 5, 4), ((0,), 1, 1, 4, 3),
                 ((0,), 1, 63, 3, 2), ((0,), 1, 63, 2, 1), ((0,), 1, 63, 1, 0), ((1,), 1, 63, 0, 0),
                 ((2,), 1, 10, 0, 1), ((2,), 11, 63, 0, 0), ((2,), 1, 10, 1, 0)]


def writer_files(f, port):
    """name -> file: the writer's non-interleaved and progressive variants of baseline file f."""
    o = port.decode(f, entropy_only=True)
    g = o["geometry"]
    color = g["ncomp"] == 3
    default = mw.DEFAULT_SCRIPT_COLOR if color else mw.DEFAULT_SCRIPT_GRAY
    custom = CUSTOM_SCRIPT if color else [((0,), *r) for comps, *r in CUSTOM_SCRIPT if comps == (0,)]
    n = len(custom)
    return {
        "non_interleaved": mw.write_non_interleaved(f, o["coef"], g),
        "non_interleaved_dri3": mw.write_non_interleaved(f, o["coef"], g, 3),
        "default": mw.write_multiscan(f, o["coef"], g, default),
        "custom": mw.write_multiscan(f, o["coef"], g, custom),
        # restarts inside EOB runs, and a DRI that changes between scans
        "custom_dri": mw.write_multiscan(f, o["coef"], g, custom, restarts=[(k % 3) * 2 for k in range(n)]),
    }


WRITER_CASES = ["420_37x53_q75", "444_64x48_q85", "422_100x70_ri3", "440_61x35_ri3", "gray_33x9_ri4", "420_flat128",
                "420_noise_q100"]


@pytest.mark.parametrize("case", WRITER_CASES)
def test_writer_files_decode_like_twin_in_pillow(hjd, port, case):
    f = small_cases()[case]
    want = np.asarray(Image.open(io.BytesIO(f)).convert("RGB"))
    for name, b in writer_files(f, port).items():
        got = np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))
        assert np.array_equal(got, want), name
        single = name.startswith("non_interleaved") and case.startswith("gray")   # one scan: a baseline file
        assert hjd.probe(b)[0] == (0 if single else -3), name
        st, o = hjd.probe(b, hjd.FLAG_MULTI_SCAN)
        assert st == 0, name
        assert (o.width, o.height) == (want.shape[1], want.shape[0])


def _rewrite_sos(f: bytes, index: int, header: bytes) -> bytes:
    """File f with the header of its index-th SOS replaced."""
    i, n = 2, 0
    while True:
        m = f[i + 1]
        ln = struct.unpack(">H", f[i + 2:i + 4])[0]
        if m == 0xDA:
            if n == index:
                return f[:i] + _seg(0xDA, header) + f[i + 2 + ln:]
            n += 1
            # skip the entropy-coded segment
            j = i + 2 + ln
            while not (f[j] == 0xFF and f[j + 1] not in (0x00,) and not 0xD0 <= f[j + 1] <= 0xD7):
                j += 1
            i = j
            continue
        i += 2 + ln


def _sos(f: bytes, index: int) -> bytes:
    i, n = 2, 0
    while True:
        m = f[i + 1]
        ln = struct.unpack(">H", f[i + 2:i + 4])[0]
        if m == 0xDA:
            if n == index:
                return f[i + 4:i + 2 + ln]
            n += 1
            j = i + 2 + ln
            while not (f[j] == 0xFF and f[j + 1] != 0x00 and not 0xD0 <= f[j + 1] <= 0xD7):
                j += 1
            i = j
            continue
        i += 2 + ln


def test_scan_header_rules(hjd):
    """T.81 G.1.1.1: each violation is HJD_IMG_ERR_UNSUPPORTED with the flag (and without it)."""
    prog, _ = PAIRS["420_37x53"]()
    flag = hjd.FLAG_MULTI_SCAN
    assert hjd.probe(prog, flag)[0] == 0

    def with_params(index, ss, se, ahal, comps=None):
        h = _sos(prog, index)
        ns = h[0]
        body = h[1:1 + 2 * ns] if comps is None else comps
        return _rewrite_sos(prog, index, bytes([len(body) // 2]) + body + bytes([ss, se, ahal]))

    bad = {
        "dc_scan_with_se": with_params(0, 0, 5, 0x01),
        "ac_scan_two_components": with_params(1, 1, 5, 0x02, _sos(prog, 0)[1:5]),
        "ac_se_below_ss": with_params(1, 6, 5, 0x02),
        "ac_se_past_63": with_params(1, 1, 64, 0x02),
        "al_past_13": with_params(1, 1, 5, 0x0E),
        "refine_wrong_ah": with_params(5, 1, 63, 0x31),       # Y 1..63 coded with Al 2: Ah must be 2
        "refine_skipping_a_bit": with_params(5, 1, 63, 0x20),  # Al must be Ah - 1
        "first_pass_twice": with_params(4, 1, 63, 0x02),      # Y 1..5 already coded by scan 1
    }
    # a refinement with no first pass before it: Cr's AC refinement moved ahead of its first pass
    bad["refine_before_first_pass"] = with_params(2, 1, 63, 0x10)
    for name, b in bad.items():
        assert hjd.probe(b, flag)[0] == -3, name
        assert hjd.probe(b)[0] == -3, name
    # sequential: every component exactly once
    _, base = PAIRS["420_37x53"]()
    from oracle import port
    port.build()
    o = port.decode(base, entropy_only=True)
    script = [((0,), 0, 63, 0, 0), ((1,), 0, 63, 0, 0), ((1,), 0, 63, 0, 0)]
    twice = mw.write_multiscan(base, o["coef"], o["geometry"], script, progressive=False)
    assert hjd.probe(twice, flag)[0] == -3
    bad_seq = mw.write_multiscan(base, o["coef"], o["geometry"], [((0,), 0, 63, 0, 0), ((1,), 0, 62, 0, 0)],
                                 progressive=False)
    assert hjd.probe(bad_seq, flag)[0] == -3
    ok_seq = mw.write_multiscan(base, o["coef"], o["geometry"], [((0,), 0, 63, 0, 0), ((1, 2), 0, 63, 0, 0)],
                                progressive=False)
    assert hjd.probe(ok_seq, flag)[0] == 0
    assert hjd.probe(ok_seq)[0] == -3


def test_scan_cap(hjd, port):
    _, base = pil_pair(synth_rgb(16, 16, 11), gray=True)
    o = port.decode(base, entropy_only=True)
    # DC, then coefficient 1 first at Al 13 and refined down to Al 0 (14 scans), the same for 2, ...: past the cap
    script = [((0,), 0, 0, 0, 0)]
    k = 1
    while len(script) < 257:
        script.append(((0,), k, k, 0, 13))
        for al in range(12, -1, -1):
            script.append(((0,), k, k, al + 1, al))
        k += 1
    at_cap = mw.write_multiscan(base, o["coef"], o["geometry"], script[:256])
    over = mw.write_multiscan(base, o["coef"], o["geometry"], script[:257])
    assert hjd.probe(at_cap, hjd.FLAG_MULTI_SCAN)[0] == 0
    assert len(hjd.scans(at_cap)) == 256
    assert hjd.probe(over, hjd.FLAG_MULTI_SCAN)[0] == -3


def test_truncated_files_keep_their_scans(hjd):
    prog, _ = PAIRS["420_37x53"]()
    sc = hjd.scans(prog)
    # cut after 3 whole scans (EOI missing), and in the middle of the 4th scan
    ends = []
    i, n = 2, 0
    while len(ends) < 4:
        m = prog[i + 1]
        ln = struct.unpack(">H", prog[i + 2:i + 4])[0]
        i += 2 + ln
        if m == 0xDA:
            ends.append(i + sc[n]["bytes"])
            i = ends[-1]
            n += 1
    st, _ = hjd.probe(prog[:ends[2]], hjd.FLAG_MULTI_SCAN)
    assert st == 0 and len(hjd.scans(prog[:ends[2]])) == 3
    mid = prog[:ends[3] - sc[3]["bytes"] // 2]
    assert hjd.probe(mid, hjd.FLAG_MULTI_SCAN)[0] == 0 and len(hjd.scans(mid)) == 4
    assert hjd.probe(prog[:20], hjd.FLAG_MULTI_SCAN)[0] == -2
