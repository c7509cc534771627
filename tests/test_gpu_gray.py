"""Luma-only decode on the GPU (FLAG_GRAY_OUT: hjd_k_luma in csrc/kernels.cu, hjd_k_mcu_scaled in csrc/scaled.cu), byte
for byte against the oracle's Y plane cropped to W x H, a KEEP_PLANES batch's Y plane, the reference's own plane tap where
it is built, and the luma of the scaled decode; through every sampling, entropy path, grid shape and host path, and with
FLAG_MULTI_SCAN (scans without luma are not read)."""
from __future__ import annotations

import time

import numpy as np
import pytest

from tests import multiscan_writer as mw
from tests.cases import cmyk_jpeg, encode_jpeg_cv, small_cases
from tests.test_gpu_edges import idct_images, tiny_images
from tests.test_gpu_scale import c4_file, free_or_skip, past_4g, report
from tests.test_gpu_scaled import golden_files
from tests.test_gray_host import gray_ref, gray_ref_scaled
from tests.test_multiscan_host import PAIRS
from tools.gen_jpegs import encode_jpeg, make_c2, synth_rgb

pytestmark = pytest.mark.gpu

SHIFTS = [1, 2, 3]
ODD = [(1, 1), (2, 3), (7, 9), (17, 9), (9, 17), (33, 31), (61, 35), (100, 70), (127, 1), (1, 129)]


def scale_flag(hjd, shift):
    return {0: 0, 1: hjd.FLAG_SCALE_1_2, 2: hjd.FLAG_SCALE_1_4, 3: hjd.FLAG_SCALE_1_8}[shift]


def decode(hjd, files, flags, overlap=None):
    with hjd.BatchDecoder(0, flags) as dec:
        if overlap is not None:
            dec.set_overlap(overlap)
        dec.upload(files)
        dec.decode()
        st = dec.status()
        out = [dec.gray(i) if st[i] >= 0 else None for i in range(len(files))]
        meta = dict(variant=dec.idct_variant, scans=[dec.num_scans(i) for i in range(len(files))],
                    sizes=[dec.out_size(i) for i in range(len(files))], timings=dec.timings(),
                    intervals=[dec.info(i).n_intervals for i in range(len(files))])
        return st, out, meta


def y_planes(hjd, files):
    """Y plane of every image of a KEEP_PLANES batch, cropped to W x H."""
    with hjd.BatchDecoder(0, hjd.FLAG_KEEP_PLANES) as dec:
        dec.upload(files)
        dec.decode()
        st = dec.status()
        slab = dec.plane_slab()
        out = []
        for i in range(len(files)):
            if st[i] < 0:
                out.append(None)
                continue
            inf = dec.info(i)
            out.append(dec.planes(i, slab)[0][:inf.height, :inf.width].copy())
        return st, out


def odd_files():
    out = []
    for k, (w, h) in enumerate(ODD):
        for s in ("4:4:4", "4:2:2", "4:2:0"):
            out.append(encode_jpeg(synth_rgb(w, h, 40 + k), 85, s, (0, 1, 3)[k % 3]))
        out.append(encode_jpeg_cv(synth_rgb(w, h, 50 + k), 85, "440", (0, 1, 3)[k % 3]))
        out.append(encode_jpeg(synth_rgb(w, h, 60 + k), 80, gray=True, restart_blocks=(0, 2)[k % 2]))
    return out


def all_files():
    return list(small_cases().values()) + golden_files() + odd_files()


@pytest.mark.parametrize("extra", ["default", "no_selfsync", "host_scan"])
def test_every_fixture_against_the_y_plane(hjd, port, extra):
    good = all_files()
    trunc = good[3][:len(good[3]) // 2]
    files = good[:10] + [b"not a jpeg at all", trunc, cmyk_jpeg()] + good[10:]
    flags = hjd.FLAG_GRAY_OUT | {"default": 0, "no_selfsync": hjd.FLAG_NO_SELFSYNC, "host_scan": hjd.FLAG_HOST_SCAN}[extra]
    st, out, meta = decode(hjd, files, flags)
    st0, planes = y_planes(hjd, files)
    assert np.array_equal(st, st0)
    assert meta["variant"] == 8
    assert meta["timings"]["color_ms"] < 0.05             # no colour stage: the gap between two events
    for i, f in enumerate(files):
        if st[i] < 0:
            assert meta["sizes"][i] == (0, 0)
            continue
        g = port.info(f)
        assert meta["sizes"][i] == (g["width"], g["height"]) and out[i].shape == (g["height"], g["width"])
        assert np.array_equal(out[i], planes[i]), i
        if st[i] == 0:
            assert np.array_equal(out[i], gray_ref(port, f)), i


def test_against_the_reference_plane_tap(hjd, refbind):
    files = [f for f in all_files() if refbind.decode(f, variant="std")["rc"] == 0]
    assert len(files) > 40
    st, out, _ = decode(hjd, files, hjd.FLAG_GRAY_OUT)
    for i, f in enumerate(files):
        r = refbind.decode(f, variant="std")
        assert np.array_equal(out[i], r["planes"][0][:r["height"], :r["width"]]), i


def test_one_component_files_equal_channel_0_of_rgb(hjd):
    files = [f for f in all_files() if hjd.probe(f)[1].ncomp == 1]
    assert len(files) >= 12
    _, out, _ = decode(hjd, files, hjd.FLAG_GRAY_OUT)
    with hjd.BatchDecoder(0) as dec:
        dec.upload(files)
        dec.decode()
        for i in range(len(files)):
            rgb = dec.rgb(i)
            assert np.array_equal(out[i], rgb[..., 0]) and np.array_equal(rgb[..., 0], rgb[..., 2]), i


def test_idct_edge_blocks(hjd, port):
    """Both clamps and the exact re-evaluation path of hjd_idct_block, under every sampling and three DQT tables."""
    imgs = idct_images()
    names = sorted(imgs)
    files = [imgs[n] for n in names] + tiny_images()
    st, out, meta = decode(hjd, files, hjd.FLAG_GRAY_OUT)
    assert (st == 0).all(), st
    _, planes = y_planes(hjd, files)
    for i, f in enumerate(files):
        assert np.array_equal(out[i], gray_ref(port, f)), (names + ["tiny"] * 48)[i]
        assert np.array_equal(out[i], planes[i]), i


# ------------------------------------------------------------------------------------------------
# grid shapes
# ------------------------------------------------------------------------------------------------
def test_similar_sizes_2d_grid(hjd, port):
    # blocks of the largest image x images <= 4 x all blocks: the (image, CTA) grid
    files = [encode_jpeg(synth_rgb(w, h, 7 + k), 85, s, r) for k, (w, h, s, r) in
             enumerate([(640, 480, "4:2:0", 8), (600, 456, "4:4:4", 0), (632, 472, "4:2:2", 3), (608, 480, "4:2:0", 0)])]
    st, out, _ = decode(hjd, files, hjd.FLAG_GRAY_OUT, overlap=0)
    assert (st == 0).all()
    for i, f in enumerate(files):
        assert np.array_equal(out[i], gray_ref(port, f)), i


def test_large_among_thumbnails_flat_grid(hjd, port):
    big = encode_jpeg(synth_rgb(4096, 4096, 8), 85, "4:2:0", 8)
    thumbs = [encode_jpeg(synth_rgb(16 + (k % 5), 16 + (k % 7), k), 85, ("4:2:0", "4:4:4", "4:2:2")[k % 3]) for k in range(30)]
    files = thumbs[:15] + [big] + thumbs[15:]
    blocks = [-(-hjd.probe(f)[1].width // 8) * -(-hjd.probe(f)[1].height // 8) for f in files]
    assert -(-max(blocks) // 128) * 128 * len(files) > 4 * sum(blocks)            # the flat grid
    st, out, _ = decode(hjd, files, hjd.FLAG_GRAY_OUT, overlap=0)
    assert (st == 0).all()
    for i, f in enumerate(files):
        assert np.array_equal(out[i], gray_ref(port, f)), i


def test_more_than_65535_images(hjd, port):
    distinct = [encode_jpeg(synth_rgb(64, 64, 300 + s), 85, ("4:4:4", "4:2:0")[s % 2], 0) for s in range(7)]
    n = 70001
    files = [distinct[i % 7] for i in range(n)]
    free0 = free_or_skip(2e9)
    t0 = time.time()
    want = [gray_ref(port, f) for f in distinct]
    with hjd.BatchDecoder(0, hjd.FLAG_GRAY_OUT) as d:
        d.set_overlap(0)
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all()
        assert d.rgb_bytes == n * 4096
        slab = d.rgb_slab()
        for i in range(n):
            off = d.info(i).rgb_offset
            assert np.array_equal(slab[off:off + 4096].reshape(64, 64), want[i % 7]), i
        report("gray, 70,001 images", free0, t0)


def test_output_slab_past_4gib(hjd, port):
    a = c4_file("420")                    # 8192 x 8192 4:2:0: 64 MiB of gray output, 1.5 M blocks
    n = 70
    free0 = free_or_skip(n * (1.5 * 2 ** 20 * 128 + 2 * len(a) + 8192 * 8192))
    t0 = time.time()
    want = gray_ref(port, a)
    with hjd.BatchDecoder(0, hjd.FLAG_GRAY_OUT) as d:
        d.set_overlap(0)
        d.upload([a] * n)
        d.decode()
        assert (d.status() == 0).all()
        assert d.idct_variant == 8 and d.rgb_bytes > 2 ** 32
        late = past_4g(d, n, lambda i: want.nbytes)
        assert len(late) >= 2 and d.info(late[-1]).rgb_offset > 2 ** 32
        for i in late:
            assert np.array_equal(d.gray(i), want), i
        report("gray past 4 GiB", free0, t0)


# ------------------------------------------------------------------------------------------------
# scaled
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shift", SHIFTS)
def test_scaled_luma(hjd, port, shift):
    imgs = idct_images()
    files = all_files() + [imgs[n] for n in sorted(imgs)[::7]] + tiny_images()[:20]
    files.append(make_c2(3, restart=True))
    st, out, meta = decode(hjd, files, hjd.FLAG_GRAY_OUT | scale_flag(hjd, shift))
    assert (st == 0).all(), st
    assert meta["variant"] == 12
    d = 1 << shift
    for i, f in enumerate(files):
        g = port.info(f)
        assert meta["sizes"][i] == (-(-g["width"] // d), -(-g["height"] // d))
        assert np.array_equal(out[i], gray_ref_scaled(port, f, shift)), (i, shift)


# ------------------------------------------------------------------------------------------------
# multi-scan
# ------------------------------------------------------------------------------------------------
def test_progressive_twins(hjd, port):
    names = sorted(PAIRS)
    pairs = [PAIRS[n]() for n in names]
    st, out, meta = decode(hjd, [p[0] for p in pairs], hjd.FLAG_GRAY_OUT | hjd.FLAG_MULTI_SCAN)
    assert (st == 0).all(), dict(zip(names, st))
    st_b, out_b, _ = decode(hjd, [p[1] for p in pairs], hjd.FLAG_GRAY_OUT)
    for n, p, o, ob, ns in zip(names, pairs, out, out_b, meta["scans"]):
        assert np.array_equal(o, ob) and np.array_equal(o, gray_ref(port, p[1])), n
        assert ns == sum(0 in s["comp"] for s in hjd.scans(p[0])), n
    for shift in SHIFTS:
        st, out, _ = decode(hjd, [p[0] for p in pairs], hjd.FLAG_GRAY_OUT | hjd.FLAG_MULTI_SCAN | scale_flag(hjd, shift))
        assert (st == 0).all()
        for n, p, o in zip(names, pairs, out):
            assert np.array_equal(o, gray_ref_scaled(port, p[1], shift)), (n, shift)


def _non_interleaved(port, truncate_after=None, restart=0):
    twin = encode_jpeg(synth_rgb(256, 192, 11), 85, "4:2:0", 0)
    o = port.decode(twin, entropy_only=True)
    script = [((c,), 0, 63, 0, 0) for c in range(3)]
    return twin, mw.write_multiscan(twin, o["coef"], o["geometry"], script, progressive=False,
                                    restarts=[restart] * 3, truncate_after=truncate_after)


def _damage_scan(hjd, f, comp):
    """The file with 16 stuffed 0xFF bytes (128 one bits: the all-ones code, which no Huffman table has) early in the
    data of the scan of component `comp` alone."""
    sc = hjd.scans(f)
    k = next(j for j, s in enumerate(sc) if list(s["comp"]) == [comp])
    pos = -1
    for _ in range(k + 1):
        pos = f.index(b"\xff\xda", pos + 1)
    at = pos + 2 + int.from_bytes(f[pos + 2:pos + 4], "big") + 8
    assert sc[k]["bytes"] > 64
    while f[at - 1] == 0xFF:                                   # not inside a stuffed 0xFF 0x00
        at += 1
    return f[:at] + b"\xff\x00" * 16 + f[at:]


def test_non_interleaved_reads_the_luma_scan_only(hjd, port):
    twin, whole = _non_interleaved(port)
    _, cut = _non_interleaved(port, truncate_after=1)          # ends right after the Y scan
    bad = _damage_scan(hjd, whole, 2)                           # undecodable code in the Cr scan
    _, with_ri = _non_interleaved(port, restart=5)
    files = [whole, cut, bad, with_ri]
    flags = hjd.FLAG_GRAY_OUT | hjd.FLAG_MULTI_SCAN
    st, out, meta = decode(hjd, files, flags)
    assert (st == 0).all(), st
    assert meta["scans"] == [1, 1, 1, 1]
    want = gray_ref(port, twin)
    for i, o in enumerate(out):
        assert np.array_equal(o, want), i
    assert meta["intervals"] == [1, 1, 1, -(-32 * 24 // 5)]
    assert hjd.probe(with_ri, flags)[1].n_intervals == -(-32 * 24 // 5)
    # the same files decoded to RGB read every scan, and report the damage
    with hjd.BatchDecoder(0, hjd.FLAG_MULTI_SCAN) as dec:
        dec.upload(files)
        dec.decode()
        st_rgb = dec.status()
        assert [dec.num_scans(i) for i in range(4)] == [3, 1, 3, 3]
    assert st_rgb[0] == 0 and st_rgb[2] > 0 and st_rgb[2] & hjd.IMG_WARN_BAD_CODE, st_rgb
    # and damage in the luma scan is reported under gray as well
    st, _, _ = decode(hjd, [_damage_scan(hjd, whole, 0)], flags)
    assert st[0] & hjd.IMG_WARN_BAD_CODE


def test_eighth_skips_ac_and_chroma_scans(hjd, port):
    prog, base = PAIRS["420_333x217"]()
    twin, ni = _non_interleaved(port)
    files = [prog, ni]
    flags = hjd.FLAG_GRAY_OUT | hjd.FLAG_MULTI_SCAN | hjd.FLAG_SCALE_1_8
    st, out, meta = decode(hjd, files, flags)
    assert (st == 0).all()
    want_scans = [sum(0 in s["comp"] and s["ss"] == 0 for s in hjd.scans(f)) for f in files]
    assert meta["scans"] == want_scans and want_scans[1] == 1
    assert np.array_equal(out[0], gray_ref_scaled(port, base, 3))
    assert np.array_equal(out[1], gray_ref_scaled(port, twin, 3))


# ------------------------------------------------------------------------------------------------
# host paths
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shift", [0, 2])
def test_decode_host_chunks_and_multi_device(hjd, port, shift):
    files = list(small_cases().values()) + golden_files() + [make_c2(5, restart=True)] + odd_files()[:20]
    flags = hjd.FLAG_GRAY_OUT | scale_flag(hjd, shift)
    want = [gray_ref_scaled(port, f, shift) if shift else gray_ref(port, f) for f in files]
    need = sum((w.nbytes + 255) // 256 * 256 for w in want)
    arena = hjd.PinnedArena(files)
    cap = int(hjd.lib().hjd_out_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n, flags))
    assert cap == need
    for overlap, chunk_images in ((3000, 0), (1, 4)):
        with hjd.BatchDecoder(0, flags) as dec:
            dec.set_overlap(overlap)
            out = np.zeros(cap, np.uint8)
            offs, st = dec.decode_host(arena, out.ctypes.data, cap, chunk_images)
            assert (st == 0).all(), st
            assert dec.rgb_bytes == need
            for i, w in enumerate(want):
                assert np.array_equal(out[offs[i]:offs[i] + w.nbytes].reshape(w.shape), w), (overlap, i)
    n_dev = hjd.lib().hjd_device_count()
    with hjd.MultiDecoder(list(range(n_dev)) if n_dev > 1 else [0, 0], flags=flags) as md:
        assert md.out_slab_bytes(arena) == need
        out = np.zeros(need, np.uint8)
        offs, st = md.decode_host(arena, out.ctypes.data, need)
        assert (st == 0).all(), st
        for i, w in enumerate(want):
            assert np.array_equal(out[offs[i]:offs[i] + w.nbytes].reshape(w.shape), w), i
    arena.close()


def test_rejected_combinations_and_api(hjd):
    for other, name in ((hjd.FLAG_KEEP_PLANES, "HJD_FLAG_KEEP_PLANES"), (hjd.FLAG_BMP_OUT, "HJD_FLAG_BMP_OUT"),
                        (hjd.FLAG_TENSOR_CORE_IDCT, "HJD_FLAG_TENSOR_CORE_IDCT"),
                        (hjd.FLAG_CUDA_CORE_IDCT, "HJD_FLAG_CUDA_CORE_IDCT")):
        for scale in (0, hjd.FLAG_SCALE_1_4):
            h = hjd.lib().hjd_batch_create(0, hjd.FLAG_GRAY_OUT | other | scale)
            assert not h
            msg = hjd.lib().hjd_last_error().decode()
            assert "hjd_batch_create" in msg and name in msg, msg
            if not scale:
                assert "HJD_FLAG_GRAY_OUT" in msg, msg
        with pytest.raises(hjd.HjdError):
            hjd.BatchDecoder(0, hjd.FLAG_GRAY_OUT | other)
        with pytest.raises(hjd.HjdError):
            hjd.MultiDecoder([0], flags=hjd.FLAG_GRAY_OUT | other)
    files = [encode_jpeg(synth_rgb(w, h, 1), 85, "4:2:0") for w, h in ((1, 1), (17, 16), (37, 53))]
    for extra in (0, hjd.FLAG_MULTI_SCAN, hjd.FLAG_HOST_SCAN, hjd.FLAG_NO_SELFSYNC, hjd.FLAG_SCALE_1_2):
        with hjd.BatchDecoder(0, hjd.FLAG_GRAY_OUT | extra) as dec:
            dec.upload(files)
            assert dec.idct_variant == 0
            dec.decode()
            assert dec.idct_variant == (12 if extra == hjd.FLAG_SCALE_1_2 else 8)
            with pytest.raises(hjd.HjdError):
                dec.rgb(0)
            assert dec.gray(1).shape == ((8, 9) if extra == hjd.FLAG_SCALE_1_2 else (16, 17))
    with hjd.BatchDecoder(0) as dec:
        dec.upload(files)
        dec.decode()
        assert dec.idct_variant & 8 == 0
        with pytest.raises(hjd.HjdError):
            dec.gray(0)
