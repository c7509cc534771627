"""HJD_FLAG_EXIF_ORIENT on the host (no GPU): the Exif APP1 parse against Pillow and on malformed tags, a sanitized
mutation fuzz of it, the numpy model of the orientation table against PIL.ImageOps.exif_transpose, and the batch plan's
staging regions and orientation jobs.  The GPU tests (tests/test_gpu_orient.py) compare against orient_ref."""
from __future__ import annotations

import io
import json
import os
import subprocess

import numpy as np
import pytest
from PIL import Image, ImageOps

from tests import exif_writer as ew
from tests.cases import small_cases
from tests.test_batch_plan import golden_files, multiscan_files
from tools.gen_jpegs import encode_jpeg, synth_rgb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hls_jpeg_decoder_b200", "csrc")
FLAG_EXIF_ORIENT = 1 << 12
TILE = 64


# ------------------------------------------------------------------------------------------------
# the orientation table (include/hjd.h), as written; also used by tests/test_gpu_orient.py
# ------------------------------------------------------------------------------------------------
def orient_ref(a: np.ndarray, o: int) -> np.ndarray:
    """Output of orientation o for a decoded image a [H', W'] or [H', W', 3]: out(x, y) = in(...) of the table."""
    H, W = a.shape[:2]
    OH, OW = (W, H) if o >= 5 else (H, W)
    y, x = np.mgrid[0:OH, 0:OW]
    ix, iy = {1: (x, y), 2: (W - 1 - x, y), 3: (W - 1 - x, H - 1 - y), 4: (x, H - 1 - y),
              5: (y, x), 6: (y, H - 1 - x), 7: (W - 1 - y, H - 1 - x), 8: (W - 1 - y, x)}[o]
    return np.ascontiguousarray(a[iy, ix])


def exif_transpose(a: np.ndarray, o: int) -> np.ndarray:
    """PIL.ImageOps.exif_transpose of the array tagged with orientation o."""
    im = Image.fromarray(a)
    im.getexif()[0x0112] = o
    return np.asarray(ImageOps.exif_transpose(im))


@pytest.mark.parametrize("bpp", [1, 3])
@pytest.mark.parametrize("o", range(1, 9))
def test_table_equals_exif_transpose(o, bpp):
    rng = np.random.default_rng(10 * o + bpp)
    for h, w in ((1, 1), (1, 7), (9, 1), (5, 3), (17, 31), (64, 65), (129, 63)):
        a = rng.integers(0, 256, (h, w) if bpp == 1 else (h, w, 3), dtype=np.uint8)
        want = exif_transpose(a, o)
        got = orient_ref(a, o)
        assert got.shape == want.shape and np.array_equal(got, want), (o, h, w)


# ------------------------------------------------------------------------------------------------
# the parse
# ------------------------------------------------------------------------------------------------
def pil_jpeg(w=37, h=21, seed=1) -> bytes:
    buf = io.BytesIO()
    Image.fromarray(synth_rgb(w, h, seed)).save(buf, format="JPEG", quality=85)
    return buf.getvalue()


def pil_orientation(f: bytes) -> int:
    return Image.open(io.BytesIO(f)).getexif().get(0x0112, 1)


@pytest.mark.parametrize("order", ["<", ">"])
@pytest.mark.parametrize("o", range(1, 9))
def test_orientation_equals_pillow(hjd, o, order):
    base = pil_jpeg(seed=o)
    for kw in (dict(), dict(before=ew.BEFORE), dict(after=ew.AFTER), dict(before=ew.BEFORE, after=ew.AFTER),
               dict(before=ew.BEFORE, exif_ifd_orientation=3, ifd1_orientation=8)):
        f = ew.with_orientation(base, o, order=order, **kw)
        assert hjd.orientation(f) == pil_orientation(f) == o, kw
        # the header parse of a batch reads it too, and the file stays decodable as before
        st, info = hjd.probe(f)
        assert st == 0 and (info.width, info.height) == (37, 21)
    # Pillow's own Exif writer
    ex = Image.Exif()
    ex[0x0112] = o
    buf = io.BytesIO()
    Image.fromarray(synth_rgb(20, 12, o)).save(buf, format="JPEG", exif=ex.tobytes())
    assert hjd.orientation(buf.getvalue()) == pil_orientation(buf.getvalue()) == o


def test_no_exif(hjd):
    for f in list(small_cases().values()) + golden_files():
        assert hjd.orientation(f) == 1
    with pytest.raises(hjd.HjdError):
        hjd.orientation(b"not a jpeg")
    with pytest.raises(hjd.HjdError):
        hjd.orientation(b"")
    assert hjd.lib().hjd_probe_jpeg_orientation(None, 0) == -1


def _truncated_app1(base, o):
    p = ew.exif_payload(o, before=ew.BEFORE, after=ew.AFTER)
    return [ew.splice(base, ew.app1(p[:k])) for k in (0, 4, 6, 8, 13, 14, 15, 30, 45, len(p) - 5)]


def malformed(base: bytes) -> dict[str, list[bytes]]:
    o = 6
    big = ew.exif_payload(o)
    return {
        "truncated_app1": _truncated_app1(base, o),
        "ifd0_offset_past_segment": [ew.with_orientation(base, o, ifd0_offset=k) for k in
                                     (len(big) - 6 - 1, len(big) - 6, 1 << 16, 0x7FFFFFFF, 0xFFFFFFFF)],
        "entry_count_past_segment": [ew.with_orientation(base, o, entry_count=k) for k in (2, 100, 0xFFFE, 0xFFFF)],
        "bad_header": [ew.splice(base, ew.app1(b"Exif\x00\x00" + m + big[10:])) for m in (b"IM*\x00", b"II\x00*", b"MM*\x00")],
        "type_long": [ew.with_orientation(base, o, typ=ew.LONG)],
        "count_0_or_2": [ew.with_orientation(base, o, count=c) for c in (0, 2)],
        "values_0_9_65535": [ew.with_orientation(base, v) for v in (0, 9, 65535)],
        "only_in_ifd1": [ew.with_orientation(base, None, ifd1_orientation=o, before=ew.BEFORE)],
        "only_in_exif_ifd": [ew.with_orientation(base, None, exif_ifd_orientation=o, after=ew.AFTER)],
        "xmp_only": [ew.splice(base, ew.xmp_app1())],
        "exif_after_sos": [ew.after_sos(base, ew.app1(ew.exif_payload(o)))],
        "not_exif_prefix": [ew.splice(base, ew.app1(b"Exif\x00\x01" + big[6:])),
                            ew.splice(base, ew.app1(b"Exif" + big[6:]))],
    }


@pytest.mark.parametrize("case", sorted(malformed(b"\xff\xd8\xff\xd9")))
def test_malformed_tags_give_1(hjd, port, case):
    for base in (pil_jpeg(), encode_jpeg(synth_rgb(40, 24, 3), 85, "4:2:0", 2)):
        st0, info0 = hjd.probe(base)
        for f in malformed(base)[case]:
            assert hjd.orientation(f) == 1, case
            st, info = hjd.probe(f)                        # never an error: the image decodes as before
            assert st == st0 == 0 and (info.width, info.height) == (info0.width, info0.height), case


def test_first_exif_app1_wins(hjd):
    base = pil_jpeg()
    # an XMP APP1 before the Exif one is skipped
    f = ew.splice(base, ew.xmp_app1(), ew.app1(ew.exif_payload(8)))
    assert hjd.orientation(f) == pil_orientation(f) == 8
    # of two Exif APP1s the first one counts, also when it has no tag or a malformed one
    for first, want in ((3, 3), (None, 1), (0, 1)):
        f = ew.splice(base, ew.app1(ew.exif_payload(first)), ew.app1(ew.exif_payload(6)))
        assert hjd.orientation(f) == want, first
    # before the first SOS only, also in a progressive file, where the walk goes on past it
    prog = io.BytesIO()
    Image.fromarray(synth_rgb(48, 40, 2)).save(prog, format="JPEG", quality=85, progressive=True)
    prog = prog.getvalue()
    assert hjd.orientation(ew.with_orientation(prog, 7)) == 7
    sos = prog.index(b"\xff\xda")
    late = prog[:sos] + prog[sos:].replace(b"\xff\xda", ew.app1(ew.exif_payload(5)) + b"\xff\xda", 1)
    mid = prog.index(b"\xff\xda", sos + 2)
    later = prog[:mid] + ew.app1(ew.exif_payload(5)) + prog[mid:]
    assert hjd.orientation(later) == 1
    assert hjd.orientation(late) == 5                      # right before the first SOS still counts
    assert hjd.probe(ew.with_orientation(prog, 7), hjd.FLAG_MULTI_SCAN)[0] == 0


# ------------------------------------------------------------------------------------------------
# the driver: sanitized fuzz and plan
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    d = tmp_path_factory.mktemp("orient_driver")
    exe = str(d / "orient_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
                           "-pthread", "-o", exe, os.path.join(ROOT, "tests", "orient_driver.cpp"),
                           os.path.join(CSRC, "batch_plan.cpp"), os.path.join(CSRC, "jpeg_parse.cpp")])
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0:abort_on_error=0", UBSAN_OPTIONS="print_stacktrace=1")

    def run(*args, files=()):
        paths = []
        for k, f in enumerate(files):
            paths.append(str(d / f"{len(os.listdir(d))}_{k}.jpg"))
            with open(paths[-1], "wb") as fh:
                fh.write(f)
        r = subprocess.run([exe] + [str(a) for a in args] + paths, capture_output=True, text=True, env=env)
        assert r.returncode == 0 and "runtime error" not in r.stderr and "Sanitizer" not in r.stderr, r.stderr[-4000:]
        return json.loads(r.stdout)
    return run


@pytest.mark.parametrize("order", ["<", ">"])
def test_fuzz_exif_payload(driver, order):
    base = ew.with_orientation(pil_jpeg(), 6, order=order, before=ew.BEFORE, after=ew.AFTER, exif_ifd_orientation=3,
                               ifd1_orientation=8)
    r = driver("fuzz", 12345 + ord(order), 2500, files=[base])
    assert sum(r["direct"]) == 2500 and r["direct"][9] == 0          # 0 (not Exif) or 1..8
    assert r["parsed"][0] == 0                                       # both walks: 1..8, and the same value
    assert r["direct"][6] > 0 and r["direct"][1] > 0 and r["direct"][0] > 0


def scaled(v, shift):
    return -(-v // (1 << shift))


def plan_files(port):
    good = list(small_cases().values())[:12] + golden_files()[:6] + [encode_jpeg(synth_rgb(w, h, k), 85, s, r)
                                                                      for k, (w, h, s, r) in enumerate(
        [(1, 1, "4:2:0", 0), (1, 65, "4:4:4", 0), (129, 1, "4:2:0", 2), (130, 67, "4:2:2", 3)])]
    files = []
    for k, f in enumerate(good):
        o = k % 9                                          # 0: no Exif segment
        files.append(f if o == 0 else ew.with_orientation(f, o, order="<>"[k % 2]))
    files[5:5] = [b"not a jpeg", ew.with_orientation(good[0][:40], 6)]            # undecodable, one with a tag
    prog = [ew.with_orientation(f, 1 + k % 8) for k, f in enumerate(multiscan_files(port))]
    return files, prog


CONFIGS = [dict(overlap=0, chunk_images=0, chunked=0), dict(overlap=40, chunk_images=0, chunked=1),
           dict(overlap=1, chunk_images=3, chunked=1)]


@pytest.mark.parametrize("cfg", CONFIGS, ids=["overlap0", "overlap40", "chunk_images3"])
@pytest.mark.parametrize("extra", ["rgb", "gray", "quarter", "gray_eighth", "multiscan"])
def test_plan_staging_and_jobs(driver, hjd, port, extra, cfg):
    files, prog = plan_files(port)
    flags = {"rgb": 0, "gray": hjd.FLAG_GRAY_OUT, "quarter": hjd.FLAG_SCALE_1_4,
             "gray_eighth": hjd.FLAG_GRAY_OUT | hjd.FLAG_SCALE_1_8, "multiscan": hjd.FLAG_MULTI_SCAN}[extra]
    if extra == "multiscan":
        files = files[:8] + prog + files[8:]
    shift = (flags >> 9) & 3
    args = [cfg["overlap"], cfg["chunk_images"], cfg["chunked"]]
    p = driver("plan", flags | FLAG_EXIF_ORIENT, *args, files=files)
    p0 = driver("plan", flags, *args, files=files)
    assert p["rc"] == p0["rc"] == 0
    # the slab is the unflagged plan's, and every image keeps its place in it
    assert p["rgb_bytes"] == p0["rgb_bytes"] and p0["stage_bytes"] == 0 and p0["jobs"] == []
    assert [im[3] for im in p["images"]] == [im[2] for im in p0["images"]] == [im[3] for im in p0["images"]]
    assert [c[:4] for c in p["chunks"]] == [c[:4] for c in p0["chunks"]]
    oriented = [i for i, im in enumerate(p["images"]) if im[0] >= 0 and im[1] != 1]
    assert len(oriented) >= 8 and {p["images"][i][1] for i in oriented} == set(range(2, 9))
    # staging: behind rgb_bytes, 256-byte aligned, disjoint, image_out_bytes each; nothing for the other images
    ends = p["rgb_bytes"]
    for i, im in enumerate(p["images"]):
        st, o, rgb_off, out_off, w, h, nbytes = im
        assert o == hjd.orientation(files[i]) if files[i][:2] == b"\xff\xd8" else o == 1
        if i in oriented:
            assert rgb_off == ends and rgb_off % 256 == 0
            ends = rgb_off + (nbytes + 255) // 256 * 256
        else:
            assert rgb_off == out_off
        # out sizes swap for 5..8, only with the flag
        if st >= 0:
            _, info = hjd.probe(files[i], flags)
            sw, sh = scaled(info.width, shift), scaled(info.height, shift)
            assert (w, h) == ((sh, sw) if o >= 5 else (sw, sh)), i
            assert p0["images"][i][4:6] == [sw, sh]
            assert nbytes == sw * sh * (1 if flags & hjd.FLAG_GRAY_OUT else 3)
    assert ends == p["rgb_bytes"] + p["stage_bytes"]
    # jobs: exactly the oriented images, in order, each inside its chunk; the tile prefix
    assert [(j[0], j[1], j[4]) for j in p["jobs"]] == [(p["images"][i][2], p["images"][i][3], p["images"][i][1])
                                                       for i in oriented]
    covered = []
    for img0, img1, rgb_lo, rgb_hi, oj0, oj1 in p["chunks"]:
        covered += list(range(oj0, oj1))
        assert all(img0 <= oriented[k] < img1 for k in range(oj0, oj1))
    assert covered == list(range(len(oriented)))
    assert p["tiles"][0] == 0 and len(p["tiles"]) == len(p["jobs"]) + 1 and p["tile"] == TILE
    for k, (j, i) in enumerate(zip(p["jobs"], oriented)):
        _, info = hjd.probe(files[i], flags)
        assert (j[2], j[3]) == (scaled(info.width, shift), scaled(info.height, shift))
        ow, oh = p["images"][i][4:6]
        assert p["tiles"][k + 1] - p["tiles"][k] == -(-ow // TILE) * -(-oh // TILE)


def test_create_refuses_bmp_out(hjd):
    for extra in (0, hjd.FLAG_GRAY_OUT, hjd.FLAG_KEEP_PLANES):
        assert not hjd.lib().hjd_batch_create(0, FLAG_EXIF_ORIENT | hjd.FLAG_BMP_OUT | extra)
        msg = hjd.lib().hjd_last_error().decode()
        assert "HJD_FLAG_EXIF_ORIENT" in msg and "HJD_FLAG_BMP_OUT" in msg, msg
    with pytest.raises(hjd.HjdError):
        hjd.BatchDecoder(0, FLAG_EXIF_ORIENT | hjd.FLAG_BMP_OUT)
    assert hjd.FLAG_EXIF_ORIENT == FLAG_EXIF_ORIENT
