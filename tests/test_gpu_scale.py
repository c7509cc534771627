"""Batches past the 32-bit boundaries of the slabs and batch-wide index spaces (DESIGN §3, "Index limits"), and the
upload guards of the spaces a batch may not cross.

Each scenario holds its own BatchDecoder, alone on the device, and skips (saying how much it needs and how much is
free) when the device has too little free memory.  Batches repeat a few distinct files, so host memory stays at a
few GB: every comparison is one image at a time, against the oracle's result for that image's file."""
from __future__ import annotations

import os
import struct
import time

import numpy as np
import pytest

from tests import multiscan_writer as mw
from tests import scaled_port as sp
from tests.test_gpu_configs import _cached
from tests.test_multiscan_host import PAIRS
from tools.gen_jpegs import encode_jpeg, synth_rgb

pytestmark = pytest.mark.gpu

GB = 1e9
C4_BLOCKS = 3 * 1024 * 1024          # 8192x8192 4:4:4
C4_RGB = 8192 * 8192 * 3
SCAN_TILE = 2048                     # elements per tile of hjd_scan_u32 (selfsync.cu)
HERE = os.path.dirname(os.path.abspath(__file__))


def free_or_skip(need: float) -> int:
    import torch
    free, _ = torch.cuda.mem_get_info(0)
    want = need + 4 * GB
    if free < want:
        pytest.skip(f"needs {want / GB:.1f} GB of free device memory ({need / GB:.1f} GB + 4 GB margin); {free / GB:.1f} GB free")
    return free


def report(name: str, free0: int, t0: float) -> None:
    import torch
    free, _ = torch.cuda.mem_get_info(0)
    print(f"\n[scale] {name}: {(free0 - free) / GB:.1f} GB of device memory, {time.time() - t0:.1f} s")


_pixels = {}


def c4_file(kind: str) -> bytes:
    """8192x8192 images of one seeded picture: "444" is make_c4 (restart-free, kernel 1b), "444_ri8" the same
    coefficients with restart markers every 8 MCUs (kernel 1a), "420" a 4:2:0 encoding."""
    def px():
        if "rgb" not in _pixels:
            _pixels["rgb"] = synth_rgb(8192, 8192, 4)
        return _pixels["rgb"]
    sub, ri = {"444": ("4:4:4", 0), "444_ri8": ("4:4:4", 8), "420": ("4:2:0", 0)}[kind]
    return _cached("c4_8192" if kind == "444" else f"c4_8192_{kind}", lambda: encode_jpeg(px(), 85, sub, ri))


def noise_file() -> bytes:
    """8192x8192 4:4:4 uniform noise at q100, restart-free: a long scan per image."""
    def make():
        rgb = np.random.default_rng(77).integers(0, 256, size=(8192, 8192, 3), dtype=np.uint8)
        return encode_jpeg(rgb, 100, "4:4:4", 0)
    return _cached("noise_8192_q100", make)


def golden(name: str) -> bytes:
    return open(os.path.join(HERE, "golden", name), "rb").read()


def arena_offsets(files):
    offs, o = [], 0
    for f in files:
        offs.append(o)
        o += (len(f) + 15) // 16 * 16
    return offs, o


# ------------------------------------------------------------------------------------------------
# S1 / S1b: the coefficient slab past block 2^29 (byte 2^36)
# ------------------------------------------------------------------------------------------------
S1_IMAGES = 174          # 2^29 blocks falls inside image 170


def s1_files():
    a, b = c4_file("444"), c4_file("444_ri8")
    prog, twin = PAIRS["444_333x217"]()
    return [a if k % 2 == 0 else b for k in range(S1_IMAGES)] + [prog], (a, b, twin)


def s1_need(files, out_bytes):
    return (S1_IMAGES * C4_BLOCKS * 128 + sum(len(f) for f in files) + sum(len(f) for f in files[0:S1_IMAGES:2])
            + out_bytes)


def test_s1_coefficients_past_block_2_29(hjd, port):
    """Kernels 1a and 1b flush blocks at batch index >= 2^29 to their own place (the index was once formed in 32
    bits: such blocks overwrote images 0-3 and left their own slots stale, with a clean status)."""
    files, (a, b, twin) = s1_files()
    free0 = free_or_skip(s1_need(files, S1_IMAGES * 2048 * 2048 * 3))
    t0 = time.time()
    want_c = {id(a): port.decode(a, want_planes=False)["coef"], id(b): port.decode(b, want_planes=False)["coef"]}
    want_c[id(files[-1])] = port.decode(twin, want_planes=False)["coef"]
    want_q = {id(a): sp.decode_scaled(a, 2)["rgb"], id(b): sp.decode_scaled(b, 2)["rgb"],
              id(files[-1]): sp.decode_scaled(twin, 2)["rgb"]}
    with hjd.BatchDecoder(0, hjd.FLAG_MULTI_SCAN | hjd.FLAG_SCALE_1_4) as d:
        d.upload(files)
        d.decode()
        st = d.status()
        assert (st == 0).all(), np.nonzero(st)
        info = [d.info(i) for i in range(len(files))]
        straddle = [i for i, f in enumerate(info) if f.block_base < 2 ** 29 < f.block_base + f.n_blocks]
        assert straddle == [170], straddle
        assert all(info[i].block_base >= 2 ** 29 for i in range(171, len(files)))
        assert info[171].restart_interval == 8 and info[172].restart_interval == 0      # both entropy kernels above it
        assert d.num_scans(len(files) - 1) > 1
        for i in [0, 1, 2, 3] + list(range(170, len(files))):
            got = d.image_coefficients_direct(i)
            bad = int((got != want_c[id(files[i])]).any(axis=1).sum())
            assert bad == 0, f"image {i} (blocks from {info[i].block_base}): {bad} blocks differ"
        for i, f in enumerate(files):
            assert np.array_equal(d.rgb(i), want_q[id(f)]), i
        report("S1 (MULTI_SCAN | SCALE_1_4)", free0, t0)


@pytest.mark.parametrize("variant", ["default", "cuda_core"])
def test_s1b_full_size_kernels_read_past_block_2_29(hjd, port, variant):
    """The full-size fused kernels read the coefficients of blocks past 2^29 (and write RGB past 2^35)."""
    files, (a, b, twin) = s1_files()
    free0 = free_or_skip(s1_need(files, S1_IMAGES * C4_RGB))
    t0 = time.time()
    want = {id(a): port.decode(a, want_planes=False)["rgb"], id(b): port.decode(b, want_planes=False)["rgb"],
            id(files[-1]): port.decode(twin, want_planes=False)["rgb"]}
    flags = hjd.FLAG_MULTI_SCAN | (hjd.FLAG_CUDA_CORE_IDCT if variant == "cuda_core" else 0)
    with hjd.BatchDecoder(0, flags) as d:
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all()
        assert d.idct_variant & (2 if variant == "cuda_core" else 1)
        for i in range(170, len(files)):
            assert np.array_equal(d.rgb(i), want[id(files[i])]), i
        report(f"S1b ({variant})", free0, t0)


# ------------------------------------------------------------------------------------------------
# S2: output and plane slabs past byte 2^32
# ------------------------------------------------------------------------------------------------
S2_IMAGES = 24           # 201 MB of RGB each: images 21-23 end past 4 GiB


def past_4g(d, n, size_of):
    out = []
    for i in range(n):
        inf = d.info(i)
        if inf.rgb_offset + size_of(i) > 2 ** 32:
            out.append(i)
    return out


@pytest.mark.parametrize("case", ["default", "cuda_core", "cuda_core_flat", "bmp_tc", "bmp_cc", "planes"])
def test_s2_output_slab_past_4gib(hjd, port, case):
    a = c4_file("444")
    tiny = golden("444_1x1.jpg")
    large = list(range(S2_IMAGES))
    if case == "cuda_core_flat":
        # hjd_launch_mcu_rgb takes the flat grid when the (image, CTA) grid has more than 4x as many thread slots as
        # there are MCUs: 24 images of 2^20 MCUs and k of one MCU give 2^20 * (24 + k) > 4 * (24 * 2^20 + k) from k = 73
        files = []
        for _ in range(S2_IMAGES):
            files += [a] + [tiny] * 4
        large = [i for i in range(len(files)) if files[i] is a]
        k = len(files) - S2_IMAGES
        slots = -(-2 ** 20 // 128) * 128 * len(files)
        assert slots > 4 * (S2_IMAGES * 2 ** 20 + k) and k > 72
    else:
        files = [a] * S2_IMAGES
    flags = {"default": 0, "cuda_core": hjd.FLAG_CUDA_CORE_IDCT, "cuda_core_flat": hjd.FLAG_CUDA_CORE_IDCT,
             "bmp_tc": hjd.FLAG_BMP_OUT, "bmp_cc": hjd.FLAG_BMP_OUT | hjd.FLAG_CUDA_CORE_IDCT,
             "planes": hjd.FLAG_KEEP_PLANES}[case]
    planes = case == "planes"
    need = S2_IMAGES * (C4_BLOCKS * 128 + 2 * len(a) + C4_RGB * (2 if planes else 1))
    free0 = free_or_skip(need)
    t0 = time.time()
    o = port.decode(a, want_planes=planes)
    want_t = port.decode(tiny, want_planes=False)["rgb"]
    with hjd.BatchDecoder(0, flags) as d:
        d.set_overlap(0)                      # one chunk: the grid rules see the whole batch
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all()
        assert d.rgb_bytes > 2 ** 32
        if case in ("default", "bmp_tc"):
            assert d.idct_variant == 1
        elif not planes:
            assert d.idct_variant == 2
        bmp = flags & hjd.FLAG_BMP_OUT
        size = (lambda i: hjd.lib().hjd_batch_bmp_bytes(d._h, i) + 64) if bmp else (lambda i: d.info(i).width * d.info(i).height * 3)
        late = past_4g(d, len(files), size)
        assert late and late[-1] == len(files) - 1 and d.info(late[0]).rgb_offset < 2 ** 32 < d.info(late[-1]).rgb_offset
        for i in late:
            w = o["rgb"] if i in large else want_t
            if bmp:
                assert d.bmp(i) == hjd.encode_bmp24(w), i
            else:
                assert np.array_equal(d.rgb(i), w), i
        if planes:
            assert hjd.lib().hjd_batch_plane_bytes(d._h) > 2 ** 32
            slab = d.plane_slab()
            for i in late:
                assert d.info(i).cr_offset > 2 ** 32
                for got, w in zip(d.planes(i, slab), o["planes"]):
                    assert np.array_equal(got, w), i
            del slab
        report(f"S2 ({case})", free0, t0)


def test_s2_scaled_output_past_4gib(hjd, port):
    """FLAG_SCALE_1_2: 90 images of 8192x8192 4:2:0 (50 MB of output each, 18 GB of coefficients)."""
    a = c4_file("420")
    n = 90
    blocks = 512 * 512 * 6
    free0 = free_or_skip(n * (blocks * 128 + 2 * len(a) + 4096 * 4096 * 3))
    t0 = time.time()
    want = sp.decode_scaled(a, 1)["rgb"]
    with hjd.BatchDecoder(0, hjd.FLAG_SCALE_1_2) as d:
        d.set_overlap(0)
        d.upload([a] * n)
        d.decode()
        assert (d.status() == 0).all()
        assert d.idct_variant == 4 and d.rgb_bytes > 2 ** 32
        late = past_4g(d, n, lambda i: want.nbytes)
        assert len(late) >= 2 and d.info(late[-1]).rgb_offset > 2 ** 32
        for i in late:
            assert np.array_equal(d.rgb(i), want), i
        report("S2 (SCALE_1_2)", free0, t0)


# ------------------------------------------------------------------------------------------------
# S3: file arena and de-stuffed buffer past byte 2^32
# ------------------------------------------------------------------------------------------------
def test_s3_arena_and_destuff_past_4gib(hjd, port):
    noise = noise_file()
    k = (2 ** 32) // len(noise) + 2                     # restart-free scans past 4 GiB, the last ones wholly
    long_ri = c4_file("444_ri8")                        # restart markers, a scan far longer than 1 MB (sliced marker scan)
    small_ri = golden("444_100x70_ri8.jpg")            # restart markers, kernel 1a
    prog, twin = PAIRS["444_333x217"]()
    files = [noise] * k + [long_ri, small_ri, prog]
    offs, arena = arena_offsets(files)
    need = (k + 1) * (C4_BLOCKS * 128 + C4_RGB) + 2 * arena
    free0 = free_or_skip(need)
    t0 = time.time()
    assert offs[k - 1] > 2 ** 32
    with hjd.BatchDecoder(0, hjd.FLAG_MULTI_SCAN) as d:
        d.set_overlap(0)                                # one chunk: one prefix sum over all restart-free scans
        d.upload(files)
        d.decode()
        st = d.status()
        assert (st == 0).all(), st
        assert d.info(k - 1).n_blocks == C4_BLOCKS and d.info(k).n_intervals > 1 and d.info(k).scan_bytes > 2 ** 20
        # the kernel-1b prefix sum over 4 N + 1 counters (N sub-sequences of 128 bytes) needs the carry loop of
        # hjd_k_scan_sums (more tiles than its 1024 threads)
        n_subs = sum(-(-d.info(i).scan_bytes // 128) for i in range(k))
        assert (4 * n_subs + 1 + SCAN_TILE - 1) // SCAN_TILE > 1024
        late = [i for i in range(len(files)) if offs[i] + len(files[i]) > 2 ** 32]
        assert late[0] <= k - 2
        want = {id(noise): port.decode(noise, want_planes=False)["coef"],
                id(long_ri): port.decode(long_ri, want_planes=False)["coef"],
                id(small_ri): port.decode(small_ri, want_planes=False)["coef"],
                id(prog): port.decode(twin, want_planes=False)["coef"]}
        for i in late:
            got = d.image_coefficients_direct(i)
            bad = int((got != want[id(files[i])]).any(axis=1).sum())
            assert bad == 0, f"image {i} (arena offset {offs[i]}): {bad} blocks differ"
        report("S3 (MULTI_SCAN, overlap off)", free0, t0)


# ------------------------------------------------------------------------------------------------
# S4: more than 65,535 images (launches split in y)
# ------------------------------------------------------------------------------------------------
S4_IMAGES = 70001
S4_FILES = 7             # 65535 = 1 (mod 7): an image decoded as another one's y-slot gets another file


def s4_files():
    return [encode_jpeg(synth_rgb(64, 64, 300 + s), 85, "4:4:4", 0) for s in range(S4_FILES)]


@pytest.mark.parametrize("case", ["default", "planes", "bmp", "scale_1_2"])
def test_s4_more_than_65535_images(hjd, port, case):
    distinct = s4_files()
    files = [distinct[i % S4_FILES] for i in range(S4_IMAGES)]
    free0 = free_or_skip(3 * GB)
    t0 = time.time()
    flags = {"default": 0, "planes": hjd.FLAG_KEEP_PLANES, "bmp": hjd.FLAG_BMP_OUT, "scale_1_2": hjd.FLAG_SCALE_1_2}[case]
    oracle = [port.decode(f, want_planes=case == "planes") for f in distinct]
    if case == "scale_1_2":
        want = [sp.decode_scaled(f, 1)["rgb"] for f in distinct]
    elif case == "bmp":
        want = [hjd.encode_bmp24(o["rgb"]) for o in oracle]
    else:
        want = [o["rgb"] for o in oracle]
    with hjd.BatchDecoder(0, flags) as d:
        d.set_overlap(0)                      # one chunk of 70,001 images
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all()
        if case == "default":
            assert d.idct_variant == 2            # the CUDA-core kernel on its (image, CTA) grid: 64 MCUs per image
        slab = d.rgb_slab()
        pslab = d.plane_slab() if case == "planes" else None
        for i in range(S4_IMAGES):
            w = want[i % S4_FILES]
            off = d.info(i).rgb_offset
            if case == "bmp":
                assert slab[off + 10:off + 10 + len(w)].tobytes() == w, i
            else:
                assert np.array_equal(slab[off:off + w.nbytes].reshape(w.shape), w), i
            if pslab is not None:
                for got, p in zip(d.planes(i, pslab), oracle[i % S4_FILES]["planes"]):
                    assert np.array_equal(got, p), i
        report(f"S4 ({case})", free0, t0)


# ------------------------------------------------------------------------------------------------
# upload guards: refused with HJD_ERR_ARG before any device memory is taken
# ------------------------------------------------------------------------------------------------
def with_size(jpg: bytes, w: int, h: int) -> bytes:
    i = 2
    while True:
        m, n = jpg[i + 1], struct.unpack(">H", jpg[i + 2:i + 4])[0]
        if m in (0xC0, 0xC1, 0xC2):
            return jpg[:i + 5] + struct.pack(">HH", h, w) + jpg[i + 9:]
        i += 2 + n


def with_scan_bytes(jpg: bytes, n: int) -> bytes:
    """The same header with a restart-free scan of n zero bytes (a large file ending with EOI: never walked on the host)."""
    sos = jpg.index(b"\xff\xda")
    end = sos + 2 + struct.unpack(">H", jpg[sos + 2:sos + 4])[0]
    return jpg[:end] + bytes(n) + b"\xff\xd9"


def refused(hjd, files, flags, message):
    import ctypes
    import torch
    with hjd.BatchDecoder(0, flags) as d:
        torch.cuda.synchronize()
        free0, _ = torch.cuda.mem_get_info(0)
        arrs = [np.frombuffer(f, dtype=np.uint8) for f in files]
        ptrs = (ctypes.c_void_p * len(files))(*[x.ctypes.data for x in arrs])
        sizes = (ctypes.c_int64 * len(files))(*[x.size for x in arrs])
        rc = hjd.lib().hjd_batch_upload(d._h, ptrs, sizes, len(files))
        err = hjd.lib().hjd_last_error().decode()
        free1, _ = torch.cuda.mem_get_info(0)
        assert rc == -1 and message in err, (rc, err)          # HJD_ERR_ARG
        assert free0 - free1 < 2 ** 20, (free0, free1)


def test_guard_blocks(hjd):
    """2^32 blocks: 342 images of 16384x16384 4:4:4 (the largest frame taken, 12,582,912 blocks each) with a short
    scan; 341 of them stay below the limit."""
    big = with_size(golden("444_64x48_q85.jpg"), 16384, 16384)
    assert hjd.probe(big)[1].n_blocks == 12582912 and 341 * 12582912 < 2 ** 32 - 1 < 342 * 12582912
    refused(hjd, [big] * 342, 0, "batch exceeds 2^32 blocks")


def test_guard_destuff_chunks(hjd):
    """2^32 16-byte chunks of restart-free scan data: 65 scans of 1 GiB (each image small)."""
    f = with_scan_bytes(golden("444_64x48_q85.jpg"), 2 ** 30)
    refused(hjd, [f] * 65, 0, "2^32 16-byte chunks")


def test_guard_multiscan_work_items(hjd):
    """2^31 multi-scan work items: 2048 progressive 1024x1024 grey files of 64 single-coefficient scans with a restart
    interval of one block (2^20 work items each).  The host keeps every file's interval starts (8 GB in all) until the
    refusal, so the test needs that much host memory."""
    avail = 0
    with open("/proc/meminfo") as fh:
        for line in fh:
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    if avail < 24 * GB:
        pytest.skip(f"needs 24 GB of available host memory; {avail / GB:.1f} GB available")
    from oracle import port
    port.build()
    tmpl = encode_jpeg(np.zeros((1024, 1024, 3), np.uint8), 85, gray=True)
    o = port.decode(tmpl, entropy_only=True)
    script = [((0,), 0, 0, 0, 0)] + [((0,), k, k, 0, 0) for k in range(1, 64)]
    f = _cached("ms_items_1024_gray", lambda: mw.write_multiscan(tmpl, o["coef"], o["geometry"], script,
                                                                restarts=[1] * len(script)))
    assert [s["restart_interval"] for s in hjd.scans(f)] == [1] * 64            # 64 scans of 16,384 intervals
    refused(hjd, [f] * 2048, hjd.FLAG_MULTI_SCAN, "2^31 multi-scan work items")
