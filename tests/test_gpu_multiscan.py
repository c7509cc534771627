"""HJD_FLAG_MULTI_SCAN on the GPU: progressive and non-interleaved files decode exactly like their baseline twins
(the single-scan files with the same quantised coefficients): same coefficients, and the oracle's RGB / planes / BMP
bytes for the twin."""
from __future__ import annotations

import ctypes
import io

import numpy as np
import pytest
from PIL import Image

from tests import multiscan_writer as mw
from tests.cases import cmyk_jpeg, small_cases
from tests.multiscan_writer import coded_mask
from tests.test_multiscan_host import CUSTOM_SCRIPT, PAIRS, pil_pair, writer_files
from tools.gen_jpegs import synth_rgb

pytestmark = pytest.mark.gpu


def decode(hjd, files, flags=0):
    flags |= hjd.FLAG_MULTI_SCAN
    with hjd.BatchDecoder(0, flags) as dec:
        dec.upload(files)
        dec.decode()
        st = dec.status()
        coef = dec.coefficients()
        out = []
        for i in range(len(files)):
            if st[i] < 0:
                out.append(None)
                continue
            r = dict(coef=dec.image_coefficients(i, coef), scans=dec.num_scans(i), info=dec.info(i))
            if flags & hjd.FLAG_BMP_OUT:
                r["bmp"] = dec.bmp(i)
            else:
                r["rgb"] = dec.rgb(i)
            out.append(r)
        if flags & hjd.FLAG_KEEP_PLANES:
            slab = dec.plane_slab()
            for i, r in enumerate(out):
                if r is not None:
                    r["planes"] = dec.planes(i, slab)
        return st, out


def check_twin(port, got, twin, mask=None):
    o = port.decode(twin)
    c = o["coef"]
    if mask is None:
        assert np.array_equal(got["coef"], c)
    else:
        assert np.array_equal(got["coef"][mask], c[mask])
    assert np.array_equal(got["rgb"], o["rgb"])


def flat_pair(restart=0):
    return pil_pair(np.full((96, 128, 3), 90, np.uint8), "4:2:0", restart=restart)


TWIN_CASES = dict(PAIRS)
TWIN_CASES.update({
    "noise_q100": lambda: pil_pair(np.random.default_rng(1).integers(0, 256, (64, 64, 3), dtype=np.uint8), quality=100),
    "noise_q100_ri1": lambda: pil_pair(np.random.default_rng(1).integers(0, 256, (64, 64, 3), dtype=np.uint8), quality=100,
                                       restart=1),
    "q10": lambda: pil_pair(synth_rgb(120, 80, 3), quality=10),
    "flat_long_eobrun": flat_pair,
    "flat_ri3": lambda: flat_pair(3),
    "gradient_444": lambda: pil_pair(np.linspace(0, 255, 200 * 150 * 3).reshape(150, 200, 3).astype(np.uint8), "4:4:4"),
})


def _small_case_twins():
    out = {}
    for name, f in small_cases().items():
        g = Image.open(io.BytesIO(f))
        rgb = np.asarray(g.convert("RGB"))
        gray = g.mode == "L"
        if name.startswith("440"):
            continue                                   # cv2-only sampling: covered by PAIRS
        sub = {"444": "4:4:4", "422": "4:2:2"}.get(name[:3], "4:2:0")
        out[name] = pil_pair(rgb, sub, gray=gray, restart=3 if "_ri" in name else 0)
    return out


def test_pillow_progressive_twins(hjd, port):
    pairs = {k: v() for k, v in TWIN_CASES.items()}
    pairs.update(_small_case_twins())
    names = sorted(pairs)
    st, out = decode(hjd, [pairs[n][0] for n in names])
    assert (st == 0).all(), dict(zip(names, st))
    for n, r in zip(names, out):
        assert r["scans"] == len(hjd.scans(pairs[n][0])), n
        check_twin(port, r, pairs[n][1])


@pytest.mark.parametrize("case", ["420_37x53_q75", "444_64x48_q85", "422_100x70_ri3", "440_61x35_ri3", "gray_33x9_ri4",
                                  "420_flat128", "420_noise_q100", "444_noise_q100_ri2"])
def test_writer_files(hjd, port, case):
    f = small_cases()[case]
    variants = writer_files(f, port)
    names = sorted(variants)
    st, out = decode(hjd, [variants[n] for n in names])
    assert (st == 0).all(), dict(zip(names, st))
    mask = coded_mask(port.decode(f, entropy_only=True)["geometry"])
    for n, r in zip(names, out):
        check_twin(port, r, f, mask)


def test_cut_after_each_scan(hjd, port):
    f = small_cases()["420_37x53_q75"]
    o = port.decode(f, entropy_only=True)
    g = o["geometry"]
    script = mw.DEFAULT_SCRIPT_COLOR
    files = [mw.write_multiscan(f, o["coef"], g, script, truncate_after=k) for k in range(1, len(script) + 1)]
    st, out = decode(hjd, files)
    assert (st == 0).all(), st
    for k, r in zip(range(1, len(script) + 1), out):
        assert np.array_equal(r["coef"], mw.expected_after(o["coef"], 3, g, script, k)), k


def test_cut_mid_scan_and_damaged_refinement(hjd, port):
    prog, twin = PAIRS["420_100x70_ri2"]()
    sc = hjd.scans(prog)
    full = len(prog) - 2
    cut = prog[:full - sc[-1]["bytes"] // 2]                      # inside the last scan (a refinement)
    st, out = decode(hjd, [cut, prog])
    assert st[0] & hjd.IMG_WARN_OVERRUN
    assert st[1] == 0
    check_twin(port, out[1], twin)
    # random bytes inside the last refinement scan: a status, and the neighbours intact
    rng = np.random.default_rng(3)
    bad = bytearray(prog)
    lo = full - sc[-1]["bytes"] + 8
    bad[lo:lo + 64] = rng.integers(0, 255, 64, dtype=np.uint8).tobytes()   # no 0xFF: markers stay where they are
    st, out = decode(hjd, [prog, bytes(bad), prog])
    assert st[0] == 0 and st[2] == 0 and st[1] >= 0
    check_twin(port, out[0], twin)
    check_twin(port, out[2], twin)


def test_mixed_batch(hjd, port):
    cs = small_cases()
    from tools.gen_jpegs import encode_jpeg
    big_rf = encode_jpeg(synth_rgb(256, 192, 5), 90, "4:2:0")            # restart-free, >= 1024 scan bytes: kernel 1b
    prog, twin = PAIRS["420_100x70_ri2"]()
    prog2, twin2 = PAIRS["444_333x217"]()
    ni = writer_files(cs["444_64x48_q85"], port)["non_interleaved_dri3"]
    files = [cs["420_100x70_ri2"], prog, big_rf, b"garbage", ni, cmyk_jpeg(), prog2, cs["gray_33x9_ri4"]]
    st, out = decode(hjd, files)
    assert st[3] < 0 and st[5] < 0
    assert (np.delete(st, [3, 5]) == 0).all(), st
    with hjd.BatchDecoder(0) as dec:                   # baseline images: the same bytes as without the flag
        dec.upload(files)
        dec.decode()
        for i in (0, 2, 7):
            assert np.array_equal(dec.rgb(i), out[i]["rgb"])
            assert np.array_equal(dec.image_coefficients_direct(i), out[i]["coef"])
    check_twin(port, out[1], twin)
    check_twin(port, out[6], twin2)
    check_twin(port, out[4], cs["444_64x48_q85"])
    st_r, out_r = decode(hjd, files[::-1])
    assert np.array_equal(st_r[::-1], st)
    for a, b in zip(out, out_r[::-1]):
        assert (a is None) == (b is None)
        if a is not None:
            assert np.array_equal(a["rgb"], b["rgb"]) and np.array_equal(a["coef"], b["coef"])


@pytest.mark.parametrize("extra", ["BMP_OUT", "KEEP_PLANES", "TENSOR_CORE_IDCT", "CUDA_CORE_IDCT", "NO_SELFSYNC",
                                   "HOST_SCAN"])
def test_flag_combinations(hjd, port, extra):
    pairs = [PAIRS[n]() for n in ("420_333x217", "gray_33x9", "420_100x70_ri2", "440_cv_61x35")]
    st, out = decode(hjd, [p[0] for p in pairs], getattr(hjd, "FLAG_" + extra))
    assert (st == 0).all(), st
    for (prog, twin), r in zip(pairs, out):
        o = port.decode(twin)
        assert np.array_equal(r["coef"], o["coef"])
        if extra == "BMP_OUT":
            assert r["bmp"] == port.bmp24_bytes(o["rgb"])
        else:
            assert np.array_equal(r["rgb"], o["rgb"])
        if extra == "KEEP_PLANES":
            for a, b in zip(r["planes"], o["planes"]):
                if b is not None and a is not None:
                    assert np.array_equal(a, b)


def test_decode_host_chunks_and_multi_device(hjd):
    pairs = [v() for v in TWIN_CASES.values()]
    files = [p[0] for p in pairs] + [p[1] for p in pairs]
    st, want = decode(hjd, files)
    arena = hjd.PinnedArena(files)
    for overlap, chunk_images in ((2000, 0), (1, 3)):
        with hjd.BatchDecoder(0, hjd.FLAG_MULTI_SCAN) as dec:
            dec.set_overlap(overlap)
            cap = int(hjd.lib().hjd_out_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n, hjd.FLAG_MULTI_SCAN))
            out = np.zeros(cap, np.uint8)
            offs, st2 = dec.decode_host(arena, out.ctypes.data, cap, chunk_images)
            assert np.array_equal(st2, st)
            for i, r in enumerate(want):
                h, w = r["rgb"].shape[:2]
                assert np.array_equal(out[offs[i]:offs[i] + h * w * 3].reshape(h, w, 3), r["rgb"]), (overlap, i)
    with hjd.MultiDecoder([0, 0], flags=hjd.FLAG_MULTI_SCAN) as md:
        cap = md.out_slab_bytes(arena)
        out = np.zeros(cap, np.uint8)
        offs, st3 = md.decode_host(arena, out.ctypes.data, cap)
        assert np.array_equal(st3, st)
        for i, r in enumerate(want):
            h, w = r["rgb"].shape[:2]
            assert np.array_equal(out[offs[i]:offs[i] + h * w * 3].reshape(h, w, 3), r["rgb"]), i
    arena.close()


@pytest.mark.timeout(1800)
def test_large_images(hjd, port):
    hd = pil_pair(synth_rgb(1920, 1080, 7), "4:2:0", quality=85)
    big = pil_pair(synth_rgb(4096, 4096, 8), "4:4:4", quality=85)
    st, out = decode(hjd, [hd[0], big[0]])
    assert (st == 0).all(), st
    check_twin(port, out[0], hd[1])
    check_twin(port, out[1], big[1])
