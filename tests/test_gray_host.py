"""HJD_FLAG_GRAY_OUT on the host (no GPU): output slab sizes, the luma-scan rule of the multi-scan planner and probe, the
plan invariants with the flag, and the CPU references the GPU tests (tests/test_gpu_gray.py) compare against.

The reference of a gray decode is the Y plane of the full decode before colour conversion: the oracle's plane tap cropped
from the MCU-padded plane to W x H, and, with a scale flag, the luma tile of the scaled decode (the numpy model of
tests/test_scaled_oracle.py, which that file checks against the C restatement)."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import multiscan_writer as mw
from tests.cases import small_cases
from tests.test_batch_plan import check_plan, golden_files, multiscan_files, restart_free_files
from tests.test_multiscan_host import PAIRS
from tests.test_scaled_oracle import FILES, model_blocks, quant_tables
from tests import scaled_port as sp
from tools.gen_jpegs import encode_jpeg, make_c5, synth_rgb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hls_jpeg_decoder_b200", "csrc")
FLAG_GRAY_OUT = 1 << 11
SHIFTS = [1, 2, 3]


# ------------------------------------------------------------------------------------------------
# references (also used by tests/test_gpu_gray.py)
# ------------------------------------------------------------------------------------------------
def gray_ref(port, jpg: bytes) -> np.ndarray:
    """The oracle's Y plane cropped to W x H: uint8 [H, W]."""
    o = port.decode(jpg, want_coef=False)
    assert o["rc"] == 0
    return np.ascontiguousarray(o["planes"][0][:o["height"], :o["width"]])


def gray_ref_scaled(port, jpg: bytes, shift: int) -> np.ndarray:
    """Luma of the scaled decode (the numpy model of the reduced IDCT on the oracle's coefficients), cropped to
    ceil(W/d) x ceil(H/d): uint8 [out_h, out_w].  shift 0: the full IDCT."""
    o = port.decode(jpg, entropy_only=True)
    g = o["geometry"]
    q, tq = quant_tables(jpg)
    n, d = 8 >> shift, 1 << shift
    hf, vf, mx, my = g["hf"], g["vf"], g["mcus_x"], g["mcus_y"]
    ny = hf * vf if g["ncomp"] == 3 else 1
    bpm = ny + 2 if g["ncomp"] == 3 else 1
    blocks = o["coef"].reshape(mx * my, bpm, 64)
    yb = model_blocks(blocks[:, :ny].reshape(-1, 64), np.broadcast_to(q[tq[0]], (mx * my * ny, 64)), n)
    yp = yb.reshape(my, mx, vf, hf, n, n).transpose(0, 2, 4, 1, 3, 5).reshape(my * vf * n, mx * hf * n)
    return np.ascontiguousarray(yp[:-(-g["height"] // d), :-(-g["width"] // d)])


def luma_scans(scans):
    """Indices of the scans a FLAG_GRAY_OUT | FLAG_MULTI_SCAN batch reads: those that contain the frame's first component."""
    return [k for k, s in enumerate(scans) if 0 in s["comp"]]


def scan_intervals(hjd, jpg: bytes, scan) -> int:
    """Restart intervals of one scan of a complete file, from its geometry (T.81 A.2): MCUs of an interleaved scan, blocks
    of a component's own grid for a non-interleaved one."""
    _, o = hjd.probe(jpg, hjd.FLAG_MULTI_SCAN)
    if len(scan["comp"]) > 1:
        units = o.mcus_x * o.mcus_y
    elif o.ncomp == 1 or scan["comp"][0] == 0:
        units = -(-o.width // 8) * -(-o.height // 8)
    else:
        cw, ch = -(-o.width // o.hf), -(-o.height // o.vf)
        units = -(-cw // 8) * -(-ch // 8)
    ri = scan["restart_interval"]
    return -(-units // ri) if ri else 1


def writer_files(port):
    """Non-interleaved and progressive files written by tests/multiscan_writer.py, with and without restart markers."""
    out = []
    for name in ("420_100x70_ri2", "422_100x70_ri3", "444_100x70_ri8", "gray_33x9_ri4"):
        f = small_cases().get(name) or open(os.path.join(ROOT, "tests", "golden", name + ".jpg"), "rb").read()
        o = port.decode(f, entropy_only=True)
        script = mw.DEFAULT_SCRIPT_GRAY if o["geometry"]["ncomp"] == 1 else mw.DEFAULT_SCRIPT_COLOR
        out.append(mw.write_multiscan(f, o["coef"], o["geometry"], script))
        out.append(mw.write_non_interleaved(f, o["coef"], o["geometry"]))
        out.append(mw.write_non_interleaved(f, o["coef"], o["geometry"], restart_blocks=3))
    return out


# ------------------------------------------------------------------------------------------------
# the references
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(FILES))
def test_model_at_full_size_is_the_oracles_y_plane(port, name):
    f = FILES[name]
    if port.decode(f, entropy_only=True)["rc"] != 0:
        pytest.skip("not decodable by the oracle")
    assert np.array_equal(gray_ref_scaled(port, f, 0), gray_ref(port, f))


@pytest.mark.parametrize("shift", SHIFTS)
def test_scaled_model_equals_the_c_restatement_on_one_component_files(port, shift):
    # a one-component file's RGB is its luma in every channel (Cb = Cr = 128 is the identity)
    files = [encode_jpeg(synth_rgb(w, h, 3 + w), 85, gray=True, restart_blocks=r) for w, h, r in
             ((1, 1, 0), (17, 9, 2), (33, 64, 0), (61, 35, 5))]
    files += [FILES[n] for n in sorted(FILES) if "gray" in n]
    for f in files:
        rgb = sp.decode_scaled(f, shift)["rgb"]
        assert np.array_equal(rgb[..., 0], rgb[..., 2])
        assert np.array_equal(gray_ref_scaled(port, f, shift), rgb[..., 0])


# ------------------------------------------------------------------------------------------------
# output slab sizes
# ------------------------------------------------------------------------------------------------
def out_slab_bytes(hjd, files, flags):
    offs, o = [], 0
    for f in files:
        offs.append(o)
        o += (len(f) + 15) // 16 * 16
    arena = np.zeros(max(o, 16), np.uint8)
    for f, off in zip(files, offs):
        arena[off:off + len(f)] = np.frombuffer(f, np.uint8)
    n = len(files)
    return int(hjd.lib().hjd_out_slab_bytes(arena.ctypes.data, (ctypes.c_int64 * n)(*offs),
                                            (ctypes.c_int64 * n)(*[len(f) for f in files]), n, flags))


ODD = [(1, 1), (17, 9), (9, 17), (37, 53), (61, 35), (8, 8), (1, 1000), (1000, 1)]


@pytest.mark.parametrize("shift", [0] + SHIFTS)
def test_out_slab_bytes(hjd, shift):
    files = golden_files() + [encode_jpeg(synth_rgb(w, h, k), 85, s) for k, (w, h) in enumerate(ODD)
                              for s in ("4:2:0", "4:4:4")]
    flags = FLAG_GRAY_OUT | (shift << 9)
    d = 1 << shift
    want = 0
    for f in files:
        st, o = hjd.probe(f)
        assert st == 0
        want += (-(-o.width // d) * -(-o.height // d) + 255) // 256 * 256
    assert out_slab_bytes(hjd, files, flags) == want
    rgb = out_slab_bytes(hjd, files, shift << 9)
    assert want < rgb and out_slab_bytes(hjd, files, 0) >= rgb
    # undecodable files take no room, as in the RGB slab
    assert out_slab_bytes(hjd, files + [b"not a jpeg"], flags) == want


# ------------------------------------------------------------------------------------------------
# multi-scan: only the scans with luma are read
# ------------------------------------------------------------------------------------------------
def test_probe_counts_the_luma_scans_only(hjd, port):
    files = writer_files(port) + [p()[0] for p in PAIRS.values()]
    seen_skipped = 0
    for f in files:
        sc = hjd.scans(f)
        want_all = sum(scan_intervals(hjd, f, s) for s in sc)
        want = sum(scan_intervals(hjd, f, sc[k]) for k in luma_scans(sc))
        st, o = hjd.probe(f, hjd.FLAG_MULTI_SCAN)
        assert st == 0 and o.n_intervals == want_all
        st, o = hjd.probe(f, hjd.FLAG_MULTI_SCAN | FLAG_GRAY_OUT)
        assert st == 0 and o.n_intervals == want, [s["comp"] for s in sc]
        # with 1/8 as well: the DC scans that contain luma
        st, o = hjd.probe(f, hjd.FLAG_MULTI_SCAN | FLAG_GRAY_OUT | hjd.FLAG_SCALE_1_8)
        assert st == 0 and o.n_intervals == sum(scan_intervals(hjd, f, sc[k]) for k in luma_scans(sc) if sc[k]["ss"] == 0)
        seen_skipped += len(sc) - len(luma_scans(sc))
    assert seen_skipped > 0


@pytest.fixture(scope="module")
def gray_plan(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("gray_plan") / "plan_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-pthread", "-o", exe, os.path.join(ROOT, "tests", "plan_driver.cpp"),
                           os.path.join(CSRC, "batch_plan.cpp"), os.path.join(CSRC, "jpeg_parse.cpp")])

    def run(files, flags, overlap=1, chunk_images=0, chunked=True):
        d = tmp_path_factory.mktemp("files")
        paths = []
        for k, f in enumerate(files):
            paths.append(str(d / f"{k}.jpg"))
            with open(paths[-1], "wb") as fh:
                fh.write(f)
        import json
        out = subprocess.run([exe, str(flags), str(overlap), str(chunk_images), str(int(chunked)), "1"] + paths,
                             check=True, capture_output=True, text=True).stdout
        return json.loads(out)
    return run


CONFIGS = [dict(overlap=0, chunked=False), dict(overlap=40, chunked=True), dict(overlap=1, chunked=True, chunk_images=3)]


@pytest.mark.parametrize("cfg", CONFIGS, ids=["overlap0", "overlap40", "chunk_images3"])
@pytest.mark.parametrize("case", ["golden", "c5", "restart_free", "multiscan", "multiscan_eighth"])
def test_plan_invariants_with_gray(gray_plan, hjd, port, case, cfg):
    flags = FLAG_GRAY_OUT
    if case == "golden":
        files = golden_files()
    elif case == "c5":
        files = [make_c5(i) for i in range(12)] + [make_c5(i, restart=False) for i in range(12, 16)]
    elif case == "restart_free":
        files = restart_free_files()
    else:
        flags |= hjd.FLAG_MULTI_SCAN | (hjd.FLAG_SCALE_1_8 if case == "multiscan_eighth" else 0)
        files = multiscan_files(port) + writer_files(port) + [golden_files()[0]]
    p = gray_plan(files, flags, **cfg)
    check_plan(p, files, flags, hjd)
    # the same plan as without the flag, apart from the multi-scan work
    p0 = gray_plan(files, flags & ~FLAG_GRAY_OUT, **cfg)
    assert p["work"] == p0["work"] and p["segs"] == p0["segs"] and p["sswork"] == p0["sswork"]
    if "multiscan" not in case:
        assert p["scans"] == p0["scans"] == [] and p["images"] == p0["images"]
        return
    # multi-scan images: their scans and work items are exactly the luma-bearing scans' (1/8: the DC ones of them)
    scans_of = {}
    for s in p["scans"]:
        scans_of.setdefault(s[0], []).append(s)
    items_of = {}
    for w in p["mswork"]:
        items_of[p["scans"][w[0]][0]] = items_of.get(p["scans"][w[0]][0], 0) + 1
    n_skipped = 0
    for i, (f, im) in enumerate(zip(files, p["images"])):
        if not im[19]:
            continue
        sc = hjd.scans(f)
        read = [k for k in luma_scans(sc) if not (case == "multiscan_eighth" and sc[k]["ss"] > 0)]
        n_skipped += len(sc) - len(read)
        assert im[18] == len(read) == len(scans_of.get(i, [])), i
        want_items = sum(scan_intervals(hjd, f, sc[k]) for k in read)
        assert im[17] == items_of.get(i, 0) == want_items, i
        assert [s[2] for s in scans_of.get(i, [])] == [scan_intervals(hjd, f, sc[k]) for k in read], i
    assert n_skipped > 0
