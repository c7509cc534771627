"""GPU tests added in round 2 (pytest -m gpu, through the C ABI): inputs beyond the reference
(SURVEY.md 8(f) rank 4), the advisor's crafted-table case, per-device kernel attributes, the honoured
chunk_images argument."""
import os

import numpy as np
import pytest

from tests import cases
from tests import jpeg_writer as jw

pytestmark = pytest.mark.gpu


def six_table_image(port, name="420_100x70_ri2", restart_interval=2):
    """A colour image whose three components select three DC and three AC tables (ids 0, 1, 2): six tables
    in shared memory, which is more than the default 48 KB window of the entropy kernels."""
    src = cases.small_cases()[name]
    o = port.decode(src, entropy_only=True)
    segs, _ = jw.segments(src)
    t = jw.dht_tables(segs)
    tables = {(0, 2): t[(0, 1)], (1, 2): t[(1, 1)]}
    sos = bytes([3, 1, 0x00, 2, 0x11, 3, 0x22, 0, 63, 0])
    return jw.rewrite(src, o["coef"], o["geometry"], tables=tables, restart_interval=restart_interval, sos_override=sos), src


def test_sixteen_bit_dc_code(hjd, port):
    """A legal 16-bit DC code (hand-built DHT): the reference searches k = 1..15 only (loadjpg.cpp:562) and
    cannot decode the file -- a deliberate deviation; the oracle's k <= 16 switch is the checker.
    Restart-marker path, restart-free path (kernel 1b) and the single-thread path."""
    src = cases.small_cases()["420_100x70_ri2"]
    o = port.decode(src)
    big = cases.small_cases()["444_gradient_q95"]
    ob = port.decode(big)
    t16 = {(0, 0): (jw.DC16_BITS, jw.DC16_VALS)}
    files = [jw.rewrite(src, o["coef"], o["geometry"], tables=t16, restart_interval=2),
             jw.rewrite(src, o["coef"], o["geometry"], tables=t16, restart_interval=0),
             jw.rewrite(big, ob["coef"], ob["geometry"], tables=t16, restart_interval=0)]
    want = [o, o, ob]
    assert hjd.probe(files[2])[1].scan_bytes >= 1024            # long enough for kernel 1b
    for flags in (0, hjd.FLAG_NO_SELFSYNC):
        with hjd.BatchDecoder(0, flags) as d:
            d.upload(files)
            d.decode()
            assert (d.status() == 0).all(), d.status()
            coef = d.coefficients()
            for i, w in enumerate(want):
                assert np.array_equal(d.image_coefficients(i, coef), w["coef"]), (flags, i)
                assert np.array_equal(d.rgb(i), w["rgb"]), (flags, i)
    try:                                                        # and the oracle, with its deviation switch, agrees
        port.set_dc16(True)
        for f, w in zip(files, want):
            assert np.array_equal(port.decode(f)["rgb"], w["rgb"])
    finally:
        port.set_dc16(False)


@pytest.mark.timeout(120)
def test_ac_table_that_never_advances_terminates(hjd, port):
    """ADVICE r1 (high): a DHT in which every AC code is a size-0 symbol with a run other than 0 / 15 never
    completes a block; the reference spins forever (loadjpg.cpp:700-829).  Every kernel must return, flag the
    image, leave good neighbours alone and produce output that depends on the input alone."""
    from tools.gen_jpegs import encode_jpeg, synth_rgb
    good = cases.small_cases()["420_64x48_q85"]
    stuck = {(1, 0): (jw.STUCK_AC_BITS, jw.STUCK_AC_VALS), (1, 1): (jw.STUCK_AC_BITS, jw.STUCK_AC_VALS)}
    free = jw.replace_tables(encode_jpeg(synth_rgb(320, 240, 61), 90, "4:2:0"), stuck)           # kernel 1b
    rst = jw.replace_tables(encode_jpeg(synth_rgb(320, 240, 62), 90, "4:2:0", restart_blocks=4), stuck)   # kernel 1a
    big = jw.replace_tables(encode_jpeg(cases.noise_rgb(512, 512, 63), 95, "4:4:4"), stuck)      # many sub-sequences
    assert hjd.probe(free)[1].scan_bytes > 4096
    want = port.decode(good)["rgb"]
    for flags in (0, hjd.FLAG_NO_SELFSYNC):
        with hjd.BatchDecoder(0, flags) as d:
            outs = []
            for rep in range(2):
                d.upload([big, good, good])                     # different slab contents in between
                d.decode()
                d.status()
                files = [good, free, rst, big, good]
                d.upload(files)
                d.decode()
                st = d.status()
                assert st[0] == 0 and st[4] == 0, st
                assert st[1] > 0 and st[2] > 0 and st[3] > 0, st
                assert np.array_equal(d.rgb(0), want) and np.array_equal(d.rgb(4), want)
                outs.append((st.copy(), d.coefficients().copy()))
            assert np.array_equal(outs[0][0], outs[1][0])
            assert np.array_equal(outs[0][1], outs[1][1])


def test_trailer_after_eoi_is_not_entropy_data(hjd, port):
    """ADVICE r1: bytes after EOI (padding, RSTn look-alikes, a second image) raise no restart warning and do
    not change the pixels."""
    a = cases.small_cases()["420_100x70_ri2"]
    b = cases.small_cases()["444_gradient_q95"]                  # restart-free, kernel 1b
    files = [a + b"\x00" * 300 + b"\xff\xd1\xff\xd2\xff\xd3" + a, b + b"\xff\xd0" * 40 + b]
    with hjd.BatchDecoder(0) as d:
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all(), d.status()
        assert np.array_equal(d.rgb(0), port.decode(a)["rgb"])
        assert np.array_equal(d.rgb(1), port.decode(b)["rgb"])


def test_six_tables_and_every_device_of_the_process(hjd, port):
    """Function attributes are per device (ADVICE r1): six distinct Huffman tables need more than 48 KB of
    shared memory in kernel 1a, the write pass of kernel 1b always does.  One process, one batch handle per
    visible GPU, the same batch on each: identical to device 0 and to the oracle."""
    six, src = six_table_image(port)
    six_free, _ = six_table_image(port, restart_interval=0)
    big = cases.small_cases()["444_gradient_q95"]
    files = [six, big, six_free, cases.small_cases()["gray_64x64"]]
    want = [port.decode(src), port.decode(big), port.decode(src), port.decode(files[3])]
    n_dev = hjd.lib().hjd_device_count()
    ref = None
    for dev in range(n_dev):
        with hjd.BatchDecoder(dev) as d:
            d.upload(files)
            d.decode()
            assert (d.status() == 0).all(), (dev, d.status())
            coef = d.coefficients()
            for i, w in enumerate(want):
                assert np.array_equal(d.image_coefficients(i, coef), w["coef"]), (dev, i)
                assert np.array_equal(d.rgb(i), w["rgb"]), (dev, i)
            slab = d.rgb_slab().copy()
            if ref is None:
                ref = slab
            assert np.array_equal(slab, ref), dev


def test_chunk_images_is_honoured(hjd, port):
    """hjd_batch_decode_host(chunk_images = k): k images per chunk; the bytes do not depend on k."""
    files = list(cases.small_cases().values())[:11]
    arena = hjd.PinnedArena(files)
    need = hjd.rgb_slab_bytes(arena)
    outs = []
    with hjd.BatchDecoder(0) as d:
        for k in (0, 1, 2, 5, 100):
            out = np.zeros(need, dtype=np.uint8)
            offs, st = d.decode_host(arena, out.ctypes.data, need, chunk_images=k)
            assert (st == 0).all()
            outs.append(out)
        for o in outs[1:]:
            assert np.array_equal(o, outs[0])
        with pytest.raises(hjd.HjdError):
            d.decode_host(arena, outs[0].ctypes.data, need, chunk_images=-1)
    o = port.decode(files[3])
    n = o["rgb"].size
    assert np.array_equal(outs[0][int(offs[3]):int(offs[3]) + n].reshape(o["rgb"].shape), o["rgb"])
    arena.close()


def test_equal_hash_keys_do_not_share_tables(hjd, port):
    """ADVICE r1: table sets are shared by content, compared byte for byte -- not by hash alone.  Two images
    with different tables (standard vs optimised) and one pair with identical ones, interleaved."""
    from tools.gen_jpegs import encode_jpeg, synth_rgb
    a = encode_jpeg(synth_rgb(96, 64, 71), 85, "4:2:0", 4)
    b = encode_jpeg(synth_rgb(96, 64, 72), 85, "4:2:0", 4, optimize=True)
    c = encode_jpeg(synth_rgb(96, 64, 73), 40, "4:2:0", 4)     # a's Huffman tables, other quantisation tables
    files = [a, b, c, a, b, c, b, a]
    with hjd.BatchDecoder(0) as d:
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all()
        for i, f in enumerate(files):
            assert np.array_equal(d.rgb(i), port.decode(f)["rgb"]), i


def test_bmp_output_mode_is_writebmp24_byte_for_byte(hjd, port):
    """HJD_FLAG_BMP_OUT: the colour kernel's epilogue writes the file WriteBMP24 writes (openjpg.cpp:504-570):
    header, bottom-up B G R rows, row padding -- for every committed fixture (odd widths: every padding
    length), Lenna (the survey's BMP sha256) and a mixed batch on the flat grid."""
    import glob
    import hashlib
    import os
    from oracle import refbind
    gdir = os.path.join(os.path.dirname(__file__), "golden")
    files = [open(p, "rb").read() for p in sorted(glob.glob(os.path.join(gdir, "*.jpg")))]
    from tools.gen_jpegs import encode_jpeg, synth_rgb
    for w in (1, 2, 3, 5, 17, 30, 63):                          # every (3w mod 4), sub-MCU and multi-MCU widths
        files.append(encode_jpeg(synth_rgb(w, 9, 300 + w), 85, "4:2:0", 2))
        files.append(encode_jpeg(synth_rgb(w, 21, 400 + w), 85, "4:4:4"))
        files.append(encode_jpeg(synth_rgb(w, 8, 500 + w), 85, gray=True))
    lenna = refbind.lenna_path()
    if lenna:
        files.append(open(lenna, "rb").read())
    with hjd.BatchDecoder(0, hjd.FLAG_BMP_OUT) as d:
        for rep in range(2):                                    # second pass: stale slab contents underneath
            d.upload(files if rep == 0 else files[::-1])
            d.decode()
            assert (d.status() == 0).all()
            order = files if rep == 0 else files[::-1]
            for i, f in enumerate(order):
                want = port.bmp24_bytes(port.decode(f)["rgb"])
                got = d.bmp(i)
                assert len(got) == len(want), i
                assert got == want, (rep, i, d.info(i).width, d.info(i).height)
        if lenna:
            assert hashlib.sha256(d.bmp(0)).hexdigest() == "af6996f7f0cb092f8282bd661f95869d6c2c983b364d8722f6ff581eaf5d12e0"
        with pytest.raises(hjd.HjdError):
            d.rgb(0)
    with pytest.raises(hjd.HjdError):
        hjd.BatchDecoder(0, hjd.FLAG_BMP_OUT | hjd.FLAG_KEEP_PLANES)


def test_short_block_idct_variant_on_every_block_length(hjd, port):
    """The IDCT leaves out the frequencies beyond zig-zag index 20 when no lane of the warp holds any (exact:
    skipped terms are zeros).  Flat images (every block DC-only), gradients, q10 ... q100 noise and mixed
    content hit both variants, in the fused and the unfused kernel; planes and RGB stay the reference's."""
    names = ["420_flat128", "420_noise_q100", "420_noise_q10", "444_gradient_q95", "420_gradient_q50", "420_100x70_ri2",
             "gray_64x64", "444_noise_q100_ri2", "420_flat_dark_ri1", "420_white_black"]
    files = [cases.small_cases()[n] for n in names]
    for flags in (0, hjd.FLAG_KEEP_PLANES):
        with hjd.BatchDecoder(0, flags) as d:
            d.upload(files)
            d.decode()
            assert (d.status() == 0).all()
            slab = d.plane_slab() if flags else None
            for i, f in enumerate(files):
                o = port.decode(f)
                assert np.array_equal(d.rgb(i), o["rgb"]), (flags, names[i])
                if flags:
                    for a, b in zip(d.planes(i, slab), o["planes"]):
                        if a is not None:
                            assert np.array_equal(a, b), names[i]


@pytest.mark.parametrize("tensor_core", [False, True])
def test_multi_device_handle_matches_single_device(hjd, port, tensor_core):
    """hjd_multi_*: the batch cut into contiguous ranges balanced by compressed bytes, one handle + one host
    thread per device.  With one visible GPU two handles share it (the sharding, offsets and threading are
    the same); with more, every device takes part.  Every image must be exactly the single-handle result --
    including a six-table image that lands on the second handle.  tensor_core: every handle uses the tensor-core
    fused kernel (persistent CTAs that take a whole SM each, launched concurrently from the handles' host threads)."""
    n_dev = hjd.lib().hjd_device_count()
    six, src = six_table_image(port)
    base = list(cases.small_cases().values())
    files = base[:9] + [six] + base[9:16] + [six]
    arena = hjd.PinnedArena(files)
    need = hjd.rgb_slab_bytes(arena)
    ref = np.zeros(need, dtype=np.uint8)
    with hjd.BatchDecoder(0) as d:
        ref_offs, st = d.decode_host(arena, ref.ctypes.data, need)
    assert (st == 0).all()
    for devices in ([0, 0], [0, 0, 0], list(range(n_dev)) if n_dev > 1 else [0]):
        with hjd.MultiDecoder(devices, hjd.FLAG_TENSOR_CORE_IDCT if tensor_core else 0) as m:
            cap = m.out_slab_bytes(arena)
            assert cap >= need
            out = np.zeros(cap, dtype=np.uint8)
            for rep in range(2):
                offs, st = m.decode_host(arena, out.ctypes.data, cap)
                assert (st == 0).all(), (devices, st)
                for i, f in enumerate(files):
                    inf = hjd.probe(f)[1]
                    nb = inf.width * inf.height * 3
                    a = out[int(offs[i]):int(offs[i]) + nb]
                    b = ref[int(ref_offs[i]):int(ref_offs[i]) + nb]
                    assert np.array_equal(a, b), (devices, i)
    o = port.decode(src)
    i = 9
    assert np.array_equal(ref[int(ref_offs[i]):int(ref_offs[i]) + o["rgb"].size].reshape(o["rgb"].shape), o["rgb"])
    arena.close()


def test_pipelined_file_to_bmp_conversion(hjd, port, tmp_path):
    """hjd_convert_jpg_files_multi: readers -> chunked GPU decodes in BMP layout -> writers.  Small chunks force
    several chunks per worker and several workers; bad inputs do not stop the rest; bytes are WriteBMP24's."""
    names = list(cases.small_cases().keys())
    ins, outs = [], []
    for k, n in enumerate(names):
        p = tmp_path / f"{k:02d}_{n}.jpg"
        p.write_bytes(cases.small_cases()[n])
        ins.append(str(p))
        outs.append(str(tmp_path / f"{k:02d}_{n}.bmp"))
    bad = tmp_path / "bad.jpg"
    bad.write_bytes(b"this is not a jpeg")
    ins[5:5] = [str(bad), str(tmp_path / "missing.jpg")]
    outs[5:5] = [str(tmp_path / "bad.bmp"), str(tmp_path / "missing.bmp")]
    n_dev = hjd.lib().hjd_device_count()
    for devices, chunk in (([0], 2), ([0], 0), (list(range(n_dev)), 3)):
        for o in outs:
            if os.path.exists(o):
                os.remove(o)
        ok = hjd.ConvertJpgFiles(ins, outs, threads=4, devices=devices, chunk_images=chunk)
        assert ok == [1] * 5 + [0, 0] + [1] * (len(names) - 5), (devices, chunk, ok)
        k = 0
        for i, (src, dst) in enumerate(zip(ins, outs)):
            if i in (5, 6):
                assert not os.path.exists(dst)
                continue
            want = port.bmp24_bytes(port.decode(cases.small_cases()[names[k]])["rgb"])
            assert open(dst, "rb").read() == want, (devices, chunk, names[k])
            k += 1


def test_against_the_reference_itself(hjd, tmp_path):
    """VERDICT r1 (weak 2): the GPU path against the REFERENCE's own code (oracle/_ref, built from a checkout of the
    reference by oracle/build_ref.sh), not its restatement: unmodified JpegParseHeader + JpegDecodeHW
    (mode 0) for restart-free colour files, the reference's block-level code with MCU-counted restarts and
    grayscale by extension (mode 1) otherwise -- coefficients, planes, RGB and the BMP file, bit for bit.
    Without oracle/_ref, the committed fixtures among these files are checked against the answers the reference gave
    for them (tests/golden/golden.json: coefficients, planes and RGB); the generated files and the BMP need it live."""
    import hashlib
    import json
    from oracle import refbind
    from tools.gen_jpegs import encode_jpeg, make_c2, synth_rgb
    live = refbind.available("std")
    gdir = os.path.join(os.path.dirname(__file__), "golden")
    golden = json.load(open(os.path.join(gdir, "golden.json")))["cases"]

    def sha(a):
        return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()

    files = {n: open(os.path.join(gdir, n + ".jpg"), "rb").read()
             for n in ("444_64x48_q85", "422_64x48_q85", "420_37x53_q75", "420_100x70_ri2", "444_opt_ri5",
                       "440_61x35_ri3", "gray_33x9_ri4", "420_noise_q100", "420_gradient_q50", "444_1x1")}
    if live:
        files["420_512x384_q90"] = encode_jpeg(synth_rgb(512, 384, 77), 90, "4:2:0")
        files["c2_1080p_ri8"] = make_c2(5)
        files["c2_1080p_twin"] = make_c2(5, restart=False)
    names = list(files)
    with hjd.BatchDecoder(0, hjd.FLAG_KEEP_PLANES) as d1, hjd.BatchDecoder(0) as d2, hjd.BatchDecoder(0, hjd.FLAG_BMP_OUT) as d3:
        for d in (d1, d2, d3):
            d.upload([files[n] for n in names])
            d.decode()
            assert (d.status() == 0).all(), d.status()
        coef, slab = d1.coefficients(), d1.plane_slab()
        for i, n in enumerate(names):
            if not live:
                g = golden[n]
                assert sha(d1.image_coefficients(i, coef)) == g["coef_sha256"], n
                planes = [p for p in d1.planes(i, slab) if p is not None]
                assert sha(np.concatenate([p.ravel() for p in planes])) == g["planes_sha256"], n
                assert sha(d1.rgb(i)) == g["rgb_sha256"] and sha(d2.rgb(i)) == g["rgb_sha256"], n
                continue
            r = refbind.decode(files[n], mode=1)
            assert r["rc"] == 0, n
            assert np.array_equal(d1.image_coefficients(i, coef), r["coef"]), n
            for a, b in zip(d1.planes(i, slab), r["planes"]):
                if a is not None:
                    assert np.array_equal(a, b), n
            assert np.array_equal(d1.rgb(i), r["rgb"]) and np.array_equal(d2.rgb(i), r["rgb"]), n
            inf = d1.info(i)
            if inf.restart_interval == 0 and inf.ncomp == 3:          # what the unmodified reference can decode
                r0 = refbind.decode(files[n], mode=0)
                assert r0["rc"] == 0 and np.array_equal(d2.rgb(i), r0["rgb"]), n
            p = str(tmp_path / "ref.bmp")
            refbind.write_bmp24(p, r["rgb"])                           # the reference's own WriteBMP24
            assert d3.bmp(i) == open(p, "rb").read(), n
