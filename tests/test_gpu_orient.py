"""EXIF orientation on the GPU (FLAG_EXIF_ORIENT: the decode kernels into staging regions, then hjd_k_orient in
csrc/orient.cu), byte for byte against the orientation table (tests/test_orient_host.py, orient_ref) applied to the same
files decoded without the flag, and against PIL.ImageOps.exif_transpose of the oracle's RGB or Y plane; through every
output kernel, sampling, entropy path, scale, host path, and at the index limits."""
from __future__ import annotations

import time

import numpy as np
import pytest

from tests import exif_writer as ew
from tests.cases import cmyk_jpeg, encode_jpeg_cv, small_cases
from tests.test_gpu_scale import c4_file, free_or_skip, past_4g, report
from tests.test_gpu_scaled import golden_files
from tests.test_gray_host import gray_ref
from tests.test_multiscan_host import PAIRS
from tests.test_orient_host import exif_transpose, orient_ref
from tools.gen_jpegs import encode_jpeg, make_c2, synth_rgb

pytestmark = pytest.mark.gpu

ODD = [(1, 1), (1, 9), (9, 1), (2, 3), (17, 9), (9, 17), (33, 31), (61, 35), (100, 70), (127, 1), (1, 129), (130, 67)]
SHIFTS = [1, 2, 3]


def scale_flag(hjd, shift):
    return {0: 0, 1: hjd.FLAG_SCALE_1_2, 2: hjd.FLAG_SCALE_1_4, 3: hjd.FLAG_SCALE_1_8}[shift]


def decode(hjd, files, flags, overlap=None):
    """(status, outputs, meta) of one batch: outputs via rgb() or gray(), None where the parse failed."""
    with hjd.BatchDecoder(0, flags) as dec:
        if overlap is not None:
            dec.set_overlap(overlap)
        dec.upload(files)
        dec.decode()
        st = dec.status()
        get = dec.gray if flags & hjd.FLAG_GRAY_OUT else dec.rgb
        out = [get(i) if st[i] >= 0 else None for i in range(len(files))]
        meta = dict(sizes=[dec.out_size(i) for i in range(len(files))], orient=[dec.orientation(i) for i in range(len(files))],
                    offsets=[dec.info(i).rgb_offset for i in range(len(files))], rgb_bytes=dec.rgb_bytes,
                    slab=dec.rgb_slab(), timings=dec.timings(), variant=dec.idct_variant)
        if flags & hjd.FLAG_KEEP_PLANES:
            meta["planes"] = dec.plane_slab()
        return st, out, meta


def odd_files():
    out = []
    for k, (w, h) in enumerate(ODD):
        for s in ("4:4:4", "4:2:2", "4:2:0"):
            out.append(encode_jpeg(synth_rgb(w, h, 40 + k), 85, s, (0, 1, 3)[k % 3]))
        out.append(encode_jpeg_cv(synth_rgb(w, h, 50 + k), 85, "440", (0, 2)[k % 2]))
        out.append(encode_jpeg(synth_rgb(w, h, 60 + k), 80, gray=True, restart_blocks=(0, 2)[k % 2]))
    return out


def base_files():
    return list(small_cases().values()) + golden_files() + odd_files()


def tagged(files, first=1):
    """Every file with every orientation 1..8 (byte orders alternating), as one list, and the orientation of each."""
    out, os_ = [], []
    for o in range(first, 9):
        for k, f in enumerate(files):
            out.append(ew.with_orientation(f, o, order="<>"[(k + o) % 2], before=ew.BEFORE[:k % 3], after=ew.AFTER[:k % 2]))
            os_.append(o)
    return out, os_


def check(hjd, port, files, os_, flags, ref_out, st, out, meta, oracle=True):
    """Flagged outputs against the table applied to the unflagged ones (ref_out), and exif_transpose of the oracle."""
    gray = flags & hjd.FLAG_GRAY_OUT
    for i, (f, o) in enumerate(zip(files, os_)):
        assert meta["orient"][i] == o
        if st[i] < 0:
            assert out[i] is None and meta["sizes"][i] == (0, 0)
            continue
        want = orient_ref(ref_out[i], o)
        assert meta["sizes"][i] == (want.shape[1], want.shape[0]), (i, o)
        assert np.array_equal(out[i], want), (i, o)
        if oracle and st[i] == 0 and not flags & (3 << 9):      # full size: the oracle's RGB or Y plane
            src = gray_ref(port, f) if gray else port.decode(f, want_coef=False)["rgb"]
            assert np.array_equal(out[i], exif_transpose(src, o)), (i, o)


EXTRA = ["default", "no_selfsync", "host_scan", "tensor_core", "cuda_core", "keep_planes", "gray", "gray_host_scan"]


@pytest.mark.parametrize("extra", EXTRA)
def test_every_fixture_and_orientation(hjd, port, extra):
    base = base_files()
    files, os_ = tagged(base)
    flags = {"default": 0, "no_selfsync": hjd.FLAG_NO_SELFSYNC, "host_scan": hjd.FLAG_HOST_SCAN,
             "tensor_core": hjd.FLAG_TENSOR_CORE_IDCT, "cuda_core": hjd.FLAG_CUDA_CORE_IDCT,
             "keep_planes": hjd.FLAG_KEEP_PLANES, "gray": hjd.FLAG_GRAY_OUT,
             "gray_host_scan": hjd.FLAG_GRAY_OUT | hjd.FLAG_HOST_SCAN}[extra]
    st0, ref, meta0 = decode(hjd, base * 8, flags)
    st, out, meta = decode(hjd, files, flags | hjd.FLAG_EXIF_ORIENT)
    assert np.array_equal(st, st0) and (st == 0).all()
    assert meta["rgb_bytes"] == meta0["rgb_bytes"] and meta["offsets"] == meta0["offsets"]
    assert meta["variant"] == meta0["variant"]
    check(hjd, port, files, os_, flags, ref, st, out, meta, oracle=extra in ("default", "gray"))
    if extra == "keep_planes":                              # the planes stay as stored
        assert np.array_equal(meta["planes"], meta0["planes"])


@pytest.mark.parametrize("gray", [False, True])
@pytest.mark.parametrize("shift", SHIFTS)
def test_scaled(hjd, port, shift, gray):
    base = list(small_cases().values()) + golden_files()[:8] + odd_files()[::3] + [make_c2(3, restart=True)]
    files, os_ = tagged(base)
    flags = scale_flag(hjd, shift) | (hjd.FLAG_GRAY_OUT if gray else 0)
    st0, ref, meta0 = decode(hjd, base * 8, flags)
    st, out, meta = decode(hjd, files, flags | hjd.FLAG_EXIF_ORIENT)
    assert (st == 0).all() and meta["rgb_bytes"] == meta0["rgb_bytes"]
    check(hjd, port, files, os_, flags, ref, st, out, meta, oracle=False)


def test_progressive_twins(hjd, port):
    names = sorted(PAIRS)
    pairs = [PAIRS[n]() for n in names]
    prog, os_ = tagged([p[0] for p in pairs])
    for flags in (hjd.FLAG_MULTI_SCAN, hjd.FLAG_MULTI_SCAN | hjd.FLAG_GRAY_OUT, hjd.FLAG_MULTI_SCAN | hjd.FLAG_SCALE_1_2):
        st0, ref, _ = decode(hjd, [p[1] for p in pairs] * 8, flags & ~hjd.FLAG_MULTI_SCAN)   # the baseline twins
        st, out, meta = decode(hjd, prog, flags | hjd.FLAG_EXIF_ORIENT)
        assert (st == 0).all(), st
        check(hjd, port, [p[1] for p in pairs] * 8, os_, flags, ref, st, out, meta,
              oracle=not flags & hjd.FLAG_SCALE_1_2)


def test_mixed_batch(hjd, port):
    good = list(small_cases().values())[:10]
    damaged = good[7][:len(good[7]) * 2 // 3] + b"\xff\xd9"             # 100x70, Ri=2: decodes with a warning
    files = [ew.with_orientation(good[0], 6), good[1], b"not a jpeg", ew.with_orientation(good[2], 3),
             ew.with_orientation(good[3][:50], 8), ew.with_orientation(damaged, 5), cmyk_jpeg(),
             ew.with_orientation(good[4], 1), ew.with_orientation(good[5], 8), b"",
             ew.with_orientation(damaged, 2)]
    os_ = [6, 1, 1, 3, 8, 5, 1, 1, 8, 1, 2]
    untagged = [good[0], good[1], b"not a jpeg", good[2], good[3][:50], damaged, cmyk_jpeg(), good[4], good[5], b"", damaged]
    for flags in (0, hjd.FLAG_GRAY_OUT):
        st0, ref, meta0 = decode(hjd, untagged, flags)
        st, out, meta = decode(hjd, files, flags | hjd.FLAG_EXIF_ORIENT)
        assert np.array_equal(st, st0)                                  # warnings are still reported
        assert st[5] > 0 and st[10] > 0 and (st[[2, 4, 6, 9]] < 0).all()
        assert meta["rgb_bytes"] == meta0["rgb_bytes"] and meta["offsets"] == meta0["offsets"]
        check(hjd, port, files, os_, flags, ref, st, out, meta, oracle=False)
        # failed images stay zero: their regions (none, all of them 0 bytes) and every byte between the images
        slab, used = meta["slab"], np.zeros(meta["rgb_bytes"], bool)
        for i in range(len(files)):
            if st[i] >= 0:
                n = out[i].nbytes
                used[meta["offsets"][i]:meta["offsets"][i] + n] = True
        assert not slab[~used].any()


def test_large_images(hjd, port):
    files = [make_c2(7, restart=True), make_c2(8, restart=False), encode_jpeg(synth_rgb(4096, 2048, 9), 85, "4:2:0", 8),
             encode_jpeg(synth_rgb(4096, 2048, 10), 85, "4:4:4", 0)]
    tagged_files, os_ = [], []
    for k, f in enumerate(files):
        for o in (1, 3, 6, 7 - k % 2):
            tagged_files.append(ew.with_orientation(f, o))
            os_.append(o)
    base = [f for f in files for _ in range(4)]
    for flags in (0, hjd.FLAG_GRAY_OUT):
        st0, ref, meta0 = decode(hjd, base, flags)
        st, out, meta = decode(hjd, tagged_files, flags | hjd.FLAG_EXIF_ORIENT)
        assert (st == 0).all() and meta["variant"] == meta0["variant"]
        check(hjd, port, tagged_files, os_, flags, ref, st, out, meta, oracle=False)
        t, t0 = meta["timings"], meta0["timings"]
        assert t["launches"] == t0["launches"] + 1


def test_more_than_65535_images(hjd, port):
    distinct = [encode_jpeg(synth_rgb(17 + s, 9 + 2 * s, 300 + s), 85, ("4:4:4", "4:2:0")[s % 2], 0) for s in range(7)]
    n = 70001
    files = [ew.with_orientation(distinct[i % 7], 1 + i % 8) for i in range(n)]
    free0 = free_or_skip(2e9)
    t0 = time.time()
    want = {(k, o): exif_transpose(port.decode(distinct[k], want_coef=False)["rgb"], o) for k in range(7) for o in range(1, 9)}
    with hjd.BatchDecoder(0, hjd.FLAG_EXIF_ORIENT) as d:
        d.set_overlap(0)
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all()
        slab = d.rgb_slab()
        for i in range(n):
            w = want[(i % 7, 1 + i % 8)]
            off = d.info(i).rgb_offset
            assert np.array_equal(slab[off:off + w.nbytes].reshape(w.shape), w), i
        report("orient, 70,001 images", free0, t0)


def test_output_past_4gib(hjd, port):
    a = c4_file("420")                    # 8192 x 8192 4:2:0: 192 MiB of RGB, 1.5 M blocks
    n = 24
    free0 = free_or_skip(n * (1.5 * 2 ** 20 * 128 + 2 * len(a) + 2 * 3 * 8192 * 8192))
    t0 = time.time()
    rgb = port.decode(a, want_coef=False)["rgb"]
    files = [a] * (n - 2) + [ew.with_orientation(a, 6), ew.with_orientation(a, 7)]
    with hjd.BatchDecoder(0, hjd.FLAG_EXIF_ORIENT) as d:
        d.set_overlap(0)
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all()
        assert d.rgb_bytes > 2 ** 32
        late = past_4g(d, n, lambda i: rgb.nbytes)
        assert late[-2:] == [n - 2, n - 1] and d.info(n - 2).rgb_offset > 2 ** 32
        for i, o in ((n - 2, 6), (n - 1, 7)):
            assert np.array_equal(d.rgb(i), exif_transpose(rgb, o)), i
        assert np.array_equal(d.rgb(late[0]), rgb)
        report("orient past 4 GiB", free0, t0)


@pytest.mark.parametrize("flags_name", ["rgb", "gray_quarter"])
def test_decode_host_chunks_and_multi_device(hjd, port, flags_name):
    base = list(small_cases().values()) + golden_files()[:6] + [make_c2(5, restart=True)] + odd_files()[:20]
    files, os_ = tagged(base, first=5)
    files += base[:4]
    os_ += [1] * 4
    flags = {"rgb": 0, "gray_quarter": hjd.FLAG_GRAY_OUT | hjd.FLAG_SCALE_1_4}[flags_name]
    _, ref, _ = decode(hjd, base * 4 + base[:4], flags)
    want = [orient_ref(r, o) for r, o in zip(ref, os_)]
    need = sum((w.nbytes + 255) // 256 * 256 for w in want)
    arena = hjd.PinnedArena(files)
    oflags = flags | hjd.FLAG_EXIF_ORIENT
    cap = int(hjd.lib().hjd_out_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n, oflags))
    assert cap == need == int(hjd.lib().hjd_out_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n, flags))
    for overlap, chunk_images in ((3000, 0), (1, 3), (1, 7)):
        with hjd.BatchDecoder(0, oflags) as dec:
            dec.set_overlap(overlap)
            out = np.zeros(cap, np.uint8)
            offs, st = dec.decode_host(arena, out.ctypes.data, cap, chunk_images)
            assert (st == 0).all(), st
            for i, w in enumerate(want):
                assert offs[i] == dec.info(i).rgb_offset
                assert np.array_equal(out[offs[i]:offs[i] + w.nbytes].reshape(w.shape), w), (overlap, chunk_images, i)
    n_dev = hjd.lib().hjd_device_count()
    with hjd.MultiDecoder(list(range(n_dev)) if n_dev > 1 else [0, 0], flags=oflags) as md:
        assert md.out_slab_bytes(arena) == need
        out = np.zeros(need, np.uint8)
        offs, st = md.decode_host(arena, out.ctypes.data, need)
        assert (st == 0).all(), st
        for i, w in enumerate(want):
            assert np.array_equal(out[offs[i]:offs[i] + w.nbytes].reshape(w.shape), w), i
    arena.close()


def test_upright_tagged_files_change_nothing(hjd):
    base = list(small_cases().values()) + golden_files()
    files = [ew.with_orientation(f, 1) for f in base] + [ew.with_orientation(f, None, before=ew.BEFORE) for f in base]
    for extra in (0, hjd.FLAG_GRAY_OUT):
        st0, _, meta0 = decode(hjd, base * 2, extra)
        st, _, meta = decode(hjd, files, extra | hjd.FLAG_EXIF_ORIENT)
        assert np.array_equal(st, st0)
        assert np.array_equal(meta["slab"], meta0["slab"]) and meta["offsets"] == meta0["offsets"]
        assert meta["timings"]["launches"] == meta0["timings"]["launches"]


def test_without_the_flag_the_tag_is_ignored(hjd):
    base = list(small_cases().values())[:8] + odd_files()[:10]
    files, os_ = tagged(base)
    for extra in (0, hjd.FLAG_GRAY_OUT, hjd.FLAG_SCALE_1_2):
        st0, _, meta0 = decode(hjd, base * 8, extra)
        st, _, meta = decode(hjd, files, extra)
        assert np.array_equal(st, st0) and meta["orient"] == os_
        assert meta["sizes"] == meta0["sizes"] and np.array_equal(meta["slab"], meta0["slab"])
        assert meta["timings"]["launches"] == meta0["timings"]["launches"]


def test_rejected_combination(hjd):
    for extra in (0, hjd.FLAG_KEEP_PLANES):
        assert not hjd.lib().hjd_batch_create(0, hjd.FLAG_EXIF_ORIENT | hjd.FLAG_BMP_OUT | extra)
        msg = hjd.lib().hjd_last_error().decode()
        assert "HJD_FLAG_EXIF_ORIENT" in msg and "HJD_FLAG_BMP_OUT" in msg, msg
        with pytest.raises(hjd.HjdError):
            hjd.MultiDecoder([0], flags=hjd.FLAG_EXIF_ORIENT | hjd.FLAG_BMP_OUT | extra)
