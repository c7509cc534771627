"""GPU tests at the geometry of BASELINE.json's configs 3, 4 and 5 (config 1 and 2 live in
test_gpu_parity.py).  Full-size where the oracle finishes in seconds, size-independent properties
otherwise."""
import hashlib
import os
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _cached(name, make):
    path = os.path.join(tempfile.gettempdir(), f"hjd_test_{os.getuid()}_{name}.jpg")     # per user: shared temp dirs
    if not os.path.exists(path):
        data = make()
        with open(path + ".tmp", "wb") as fh:
            fh.write(data)
        os.replace(path + ".tmp", path)
    return open(path, "rb").read()


def test_config4_8192_444_restart_free(hjd, port):
    """Config 4: single 8192x8192 4:4:4 baseline JPEG with no restart markers -> kernel 1b.
    All 3,145,728 blocks of coefficients bit-exact against the oracle; RGB identical."""
    from tools.gen_jpegs import make_c4
    jpg = _cached("c4_8192", lambda: make_c4(8192, 4))
    with hjd.BatchDecoder(0) as d:
        d.upload([jpg])
        d.decode()
        assert d.status()[0] == 0
        inf = d.info(0)
        assert (inf.width, inf.height, inf.n_blocks, inf.restart_interval) == (8192, 8192, 3145728, 0)
        coef = d.coefficients()
        o = port.decode(jpg, want_planes=False)
        assert o["rc"] == 0
        bad = int((coef != o["coef"]).any(axis=1).sum())
        assert bad == 0, f"{bad} coefficient blocks differ"
        rgb = d.rgb(0)
        diff = np.abs(rgb.astype(np.int16) - o["rgb"].astype(np.int16))
        assert diff.max() <= 1, f"max RGB diff {diff.max()}"
        assert int((diff != 0).sum()) == 0, f"{int((diff != 0).sum())} RGB samples differ"
        assert 2 <= d.selfsync_rounds <= 8
        # idempotence: decoding the resident batch again gives the same bytes
        d.decode()
        assert hashlib.sha256(d.rgb(0).tobytes()).hexdigest() == hashlib.sha256(rgb.tobytes()).hexdigest()


def test_config5_thumbnails(hjd, port):
    """Config 5: 256x256 thumbnails, even = grayscale, odd = 4:2:0, q75, Ri = 8 (512 of them),
    every image checked against the oracle."""
    from tools.gen_jpegs import make_batch
    files = make_batch("c5", 512)
    with hjd.BatchDecoder(0) as d:
        d.upload(files)
        d.decode()
        assert (d.status() == 0).all()
        assert d.info(0).ncomp == 1 and d.info(1).ncomp == 3
        coef = d.coefficients()
        slab = d.rgb_slab()
        for i, f in enumerate(files):
            o = port.decode(f, want_planes=False)
            inf = d.info(i)
            assert np.array_equal(coef[inf.block_base:inf.block_base + inf.n_blocks], o["coef"]), i
            got = slab[inf.rgb_offset:inf.rgb_offset + 256 * 256 * 3].reshape(256, 256, 3)
            assert np.array_equal(got, o["rgb"]), i


def test_config3_sharding_invariance(hjd):
    """Config 3: the same batch decoded as 1, 2, 4 and 8 shards gives identical per-image bytes
    (what the multi-GPU run does with one shard per GPU; no collective involved)."""
    from hls_jpeg_decoder_b200.sharding import shard_range
    from tools.gen_jpegs import make_c2
    files = [make_c2(i, width=480, height=270) for i in range(16)]
    with hjd.BatchDecoder(0) as d:
        d.upload(files)
        d.decode()
        want = [hashlib.sha256(d.rgb(i).tobytes()).hexdigest() for i in range(len(files))]
        for world in (2, 4, 8):
            got = [None] * len(files)
            for rank in range(world):
                lo, hi = shard_range([len(f) for f in files], rank, world)
                if hi > lo:
                    d.upload(files[lo:hi])
                    d.decode()
                    assert (d.status() == 0).all()
                    for k in range(hi - lo):
                        got[lo + k] = hashlib.sha256(d.rgb(k).tobytes()).hexdigest()
            assert got == want, world
