"""Reduced-size decode on the GPU (FLAG_SCALE_1_2 / _1_4 / _1_8, csrc/scaled.cu): bit for bit the CPU
restatement hjdo_decode_scaled (tests/scaled_oracle.c), through every grid shape, sampling, table layout, entropy path and host path, and with
FLAG_MULTI_SCAN (at 1/8 only the DC scans are read)."""
from __future__ import annotations

import glob
import os

import numpy as np
import pytest

from tests import multiscan_writer as mw
from tests import scaled_port as sp
from tests.cases import cmyk_jpeg, small_cases
from tests.test_gpu_edges import idct_images, tiny_images
from tests.test_multiscan_host import PAIRS
from tools.gen_jpegs import encode_jpeg, make_c2, synth_rgb

pytestmark = pytest.mark.gpu

SHIFTS = [1, 2, 3]


def scale_flag(hjd, shift):
    return {1: hjd.FLAG_SCALE_1_2, 2: hjd.FLAG_SCALE_1_4, 3: hjd.FLAG_SCALE_1_8}[shift]


def decode(hjd, files, flags):
    with hjd.BatchDecoder(0, flags) as dec:
        dec.upload(files)
        dec.decode()
        st = dec.status()
        out = [dec.rgb(i) if st[i] >= 0 else None for i in range(len(files))]
        sizes = [dec.out_size(i) for i in range(len(files))]
        scans = [dec.num_scans(i) for i in range(len(files))]
        return st, out, dict(variant=dec.idct_variant, sizes=sizes, scans=scans)


def check(port, files, out, shift, names=None):
    for i, f in enumerate(files):
        want = sp.decode_scaled(f, shift)["rgb"]
        assert np.array_equal(out[i], want), (names[i] if names else i, shift)


def golden_files():
    return [open(p, "rb").read() for p in sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.jpg")))]


@pytest.mark.parametrize("shift", SHIFTS)
def test_mixed_batch(hjd, port, shift):
    good = list(small_cases().values()) + golden_files()
    trunc = good[3][:len(good[3]) // 2]
    files = good[:10] + [b"not a jpeg at all", trunc, cmyk_jpeg()] + good[10:]
    st0, _, _ = decode(hjd, files, 0)
    st, out, meta = decode(hjd, files, scale_flag(hjd, shift))
    assert np.array_equal(st, st0)
    assert meta["variant"] == 4
    d = 1 << shift
    for i, f in enumerate(files):
        if st[i] < 0:
            assert meta["sizes"][i] == (0, 0)
            continue
        g = port.info(f)
        assert meta["sizes"][i] == (-(-g["width"] // d), -(-g["height"] // d))
        if st[i] == 0:
            assert np.array_equal(out[i], sp.decode_scaled(f, shift)["rgb"]), (i, shift)


@pytest.mark.parametrize("shift", SHIFTS)
def test_edge_blocks_every_sampling_three_tables(hjd, port, shift):
    imgs = idct_images()
    names = sorted(imgs)
    files = [imgs[n] for n in names] + tiny_images()
    st, out, meta = decode(hjd, files, scale_flag(hjd, shift))
    assert (st == 0).all(), st
    assert meta["variant"] == 4
    check(port, files, out, shift, names + ["tiny"] * (len(files) - len(names)))


@pytest.mark.timeout(1800)
def test_large_images(hjd, port):
    files = [make_c2(3, restart=False), make_c2(3, restart=True), encode_jpeg(synth_rgb(4096, 4096, 8), 85, "4:4:4")]
    want = {s: [sp.decode_scaled(f, s)["rgb"] for f in files] for s in SHIFTS}
    for shift in SHIFTS:
        st, out, _ = decode(hjd, files, scale_flag(hjd, shift))
        assert (st == 0).all(), st
        for i in range(len(files)):
            assert np.array_equal(out[i], want[shift][i]), (i, shift)


@pytest.mark.parametrize("shift", SHIFTS)
def test_decode_host_chunks_and_multi_device(hjd, port, shift):
    files = list(small_cases().values()) + golden_files() + [make_c2(5, restart=True)]
    flags = scale_flag(hjd, shift)
    want = [sp.decode_scaled(f, shift)["rgb"] for f in files]
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
    with hjd.MultiDecoder([0, 0], flags=flags) as md:
        assert md.out_slab_bytes(arena) == need
        out = np.zeros(need, np.uint8)
        offs, st = md.decode_host(arena, out.ctypes.data, need)
        assert (st == 0).all(), st
        for i, w in enumerate(want):
            assert np.array_equal(out[offs[i]:offs[i] + w.nbytes].reshape(w.shape), w), i
    arena.close()


@pytest.mark.parametrize("shift", SHIFTS)
def test_progressive_twins(hjd, port, shift):
    names = sorted(PAIRS)
    pairs = [PAIRS[n]() for n in names]
    st, out, meta = decode(hjd, [p[0] for p in pairs], scale_flag(hjd, shift) | hjd.FLAG_MULTI_SCAN)
    assert (st == 0).all(), dict(zip(names, st))
    for n, p, o, ns in zip(names, pairs, out, meta["scans"]):
        assert np.array_equal(o, sp.decode_scaled(p[1], shift)["rgb"]), n
        sc = hjd.scans(p[0])
        assert ns == (sum(s["ss"] == 0 for s in sc) if shift == 3 else len(sc)), n


def _writer_file(port, truncate_after=None):
    f = small_cases()["420_100x70_ri2"]
    o = port.decode(f, entropy_only=True)
    return f, mw.write_multiscan(f, o["coef"], o["geometry"], mw.DEFAULT_SCRIPT_COLOR, truncate_after=truncate_after)


def test_eighth_reads_the_dc_scans_only(hjd, port):
    script = mw.DEFAULT_SCRIPT_COLOR
    dc = [k for k, s in enumerate(script) if s[1] == 0]
    twin, whole = _writer_file(port)
    _, cut = _writer_file(port, truncate_after=dc[-1] + 1)           # ends right after the last DC scan
    # random bytes at the end of the first AC scan's data, in a window with no 0xFF next to it (the markers stay where they are)
    lo, hi = len(_writer_file(port, truncate_after=1)[1]) - 2, len(_writer_file(port, truncate_after=2)[1]) - 2
    rng = np.random.default_rng(5)
    bad = bytearray(whole)
    at = next(a for a in range(hi - 40, lo, -1) if 0xFF not in whole[a - 1:a + 33])   # the scan's data ends at hi
    bad[at:at + 32] = rng.integers(0, 255, 32, dtype=np.uint8).tobytes()
    files = [whole, cut, bytes(bad)]
    flags = hjd.FLAG_MULTI_SCAN | hjd.FLAG_SCALE_1_8
    st, out, meta = decode(hjd, files, flags)
    assert (st == 0).all(), st
    assert meta["scans"] == [len(dc)] * 3
    want = sp.decode_scaled(twin, 3)["rgb"]
    for i, o in enumerate(out):
        assert np.array_equal(o, want), i
    with hjd.BatchDecoder(0, flags) as dec:                         # no restart markers: one work item per DC scan
        dec.upload(files)
        assert [dec.info(i).n_intervals for i in range(3)] == [len(dc)] * 3
        assert hjd.probe(whole, flags)[1].n_intervals == len(dc)
    # without the scale flag the damaged AC scan is read
    _, _, meta_full = decode(hjd, files, hjd.FLAG_MULTI_SCAN)
    assert meta_full["scans"] == [len(script), dc[-1] + 1, len(script)]


def test_rejected_combinations_and_out_size(hjd):
    for shift in SHIFTS:
        f = scale_flag(hjd, shift)
        for other in (hjd.FLAG_KEEP_PLANES, hjd.FLAG_BMP_OUT, hjd.FLAG_TENSOR_CORE_IDCT, hjd.FLAG_CUDA_CORE_IDCT):
            with pytest.raises(hjd.HjdError):
                hjd.BatchDecoder(0, f | other)
            with pytest.raises(hjd.HjdError):
                hjd.MultiDecoder([0], flags=f | other)
    files = [encode_jpeg(synth_rgb(w, h, 1), 85, "4:2:0") for w, h in ((1, 1), (17, 16), (37, 53), (61, 35))]
    with hjd.BatchDecoder(0, 0) as dec:
        dec.upload(files)
        assert [dec.out_size(i) for i in range(4)] == [(1, 1), (17, 16), (37, 53), (61, 35)]
    for shift in SHIFTS:
        d = 1 << shift
        st, out, meta = decode(hjd, files, scale_flag(hjd, shift))
        assert meta["sizes"] == [(-(-w // d), -(-h // d)) for w, h in ((1, 1), (17, 16), (37, 53), (61, 35))]
        assert [o.shape for o in out] == [(s[1], s[0], 3) for s in meta["sizes"]]
