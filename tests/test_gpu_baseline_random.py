"""Kernels 1a (restart intervals) and 1b (restart-free, self-synchronising) on random baseline files: random Huffman
tables of every code length and of a single code, up to four table ids per class (SOF1), table sets shared by
content under other ids, redefined ids, every restart layout, 0xFF fill bytes before RSTn and EOI, FF 00 runs at
every arena phase, and DC predictors that wrap int16.  The coefficients equal the T.81 restatement's
(tests/t81_decode.py) and the RGB the oracle's decode of the baseline twin, under every path that decodes these
files.  Also a stream that never self-synchronises: kernel 1b's synchronisation rounds have to walk a chain of
wrong entry states across the whole image, one range of sub-sequences per round.

Measured on an NVIDIA B200 (1000 W power limit), the decode of the 2992x3000 non-synchronising image (6,679
sub-sequences, one upload, wall clock around decode() and a synchronise) takes about 13 ms with 32 sub-sequences
per warp (211 ranges, 211 rounds) and about 3.6 ms with 256 (27 ranges); a restart-free photograph of that size
decodes in well under 1 ms.  A hostile file can so serialise kernel 1b: its rounds grow with the number of ranges
(the round limit, sub-sequences / 32 + 8, keeps them bounded and is never reached).  That is a known cost, not a
fault: the output stays exact."""
from __future__ import annotations

import numpy as np
import pytest

from tests import baseline_random as br
from tests import t81_decode as t81

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]

FLAG_SETS = ("default", "no_selfsync", "host_scan", "keep_planes", "cuda_core", "tensor_core")


def _flags(hjd, name):
    return {"default": 0, "no_selfsync": hjd.FLAG_NO_SELFSYNC, "host_scan": hjd.FLAG_HOST_SCAN,
            "keep_planes": hjd.FLAG_KEEP_PLANES, "cuda_core": hjd.FLAG_CUDA_CORE_IDCT,
            "tensor_core": hjd.FLAG_TENSOR_CORE_IDCT}[name]


def decode(hjd, files, flags=0, ss_range=0):
    """dict(status, rounds, coef, rgb, planes) of one batch decoded once."""
    with hjd.BatchDecoder(0, flags) as d:
        if ss_range:
            d.set_selfsync_range(ss_range)
        d.upload(files)
        d.decode()
        st = d.status().copy()
        coef = d.coefficients()
        slab = d.plane_slab() if flags & hjd.FLAG_KEEP_PLANES else None
        out = dict(status=st, rounds=d.selfsync_rounds, coef=[], rgb=[], planes=[])
        for i in range(len(files)):
            out["coef"].append(d.image_coefficients(i, coef).copy())
            out["rgb"].append(d.rgb(i).copy())
            if slab is not None:
                out["planes"].append([None if p is None else p.copy() for p in d.planes(i, slab)])
    return out


def check(batch, got, what):
    assert (got["status"] == 0).all(), (what, got["status"])
    for i, c in enumerate(batch):
        assert np.array_equal(got["coef"][i], c["t81"]), (what, i, "coefficients")
        assert np.array_equal(got["rgb"][i], c["want"]["rgb"]), (what, i, "rgb")
        for a, b in zip(got["planes"][i] if got["planes"] else [], c["want"]["planes"]):
            if a is not None:
                assert np.array_equal(a, b), (what, i, "planes")


@pytest.fixture(scope="module")
def batch(port):
    cases = []
    for i in range(br.N_BATCH):
        c = br.random_case(**br.batch_params(i), port=port)
        c["t81"] = t81.decode(c["file"])[0]
        assert np.array_equal(c["t81"], c["coef"]), i
        c["want"] = port.decode(c["twin"])
        assert c["want"]["rc"] == 0, i
        cases.append(c)
    return cases


@pytest.fixture(scope="module")
def default_decode(hjd, batch):
    return decode(hjd, [c["file"] for c in batch])


@pytest.mark.parametrize("flag_set", FLAG_SETS)
def test_random_batch(hjd, batch, default_decode, flag_set):
    got = default_decode if flag_set == "default" else decode(hjd, [c["file"] for c in batch], _flags(hjd, flag_set))
    check(batch, got, flag_set)


def test_reverse_order(hjd, batch):
    got = decode(hjd, [c["file"] for c in batch[::-1]])
    check(batch[::-1], got, "reversed")


def test_selfsync_ranges(hjd, batch):
    free = [c for c in batch if c["stats"]["n_intervals"] == 1]
    assert len(free) >= 16
    for rng in (32, 64, 128, 256):
        check(free, decode(hjd, [c["file"] for c in free], ss_range=rng), f"range {rng}")


def test_chunks_and_devices(hjd, batch):
    files = [c["file"] for c in batch]
    want = [c["want"]["rgb"] for c in batch]
    arena = hjd.PinnedArena(files)
    try:
        def check_host(offs, st, out):
            assert (st == 0).all(), st
            for i, w in enumerate(want):
                h, wd = w.shape[:2]
                assert np.array_equal(out[offs[i]:offs[i] + h * wd * 3].reshape(h, wd, 3), w), i
        with hjd.BatchDecoder(0) as dec:
            dec.set_overlap(1)
            cap = int(hjd.lib().hjd_out_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n, 0))
            out = np.zeros(cap, np.uint8)
            check_host(*dec.decode_host(arena, out.ctypes.data, cap, 3), out)
        with hjd.MultiDecoder([0, 0]) as md:
            cap = md.out_slab_bytes(arena)
            out = np.zeros(cap, np.uint8)
            check_host(*md.decode_host(arena, out.ctypes.data, cap), out)
    finally:
        arena.close()


def test_fill_bytes_long_scans(hjd, port):
    """Fill bytes before RSTn and EOI in scans shorter and longer than HJD_SCAN_WALK_MAX (64 KiB: beyond it the scan
    length is taken from the trailing EOI without walking the markers), restart and restart-free, through kernel 1a,
    kernel 1b, the host marker walk and the single-thread path: T.81's coefficients and status 0."""
    cases = []
    for k, (w, h, s, dri, fill) in enumerate([(480, 320, "4:4:4", 0, 7), (480, 320, "4:2:0", 3, 7),
                                              (480, 320, "4:4:4", 13, 1), (400, 400, "gray", 0, 2),
                                              (64, 48, "4:2:2", 0, 9), (64, 48, "4:2:2", 2, 9)]):
        c = br.random_case(9000 + k, w, h, s, dri=dri, fill=fill, wrap=False, share=False, port=port)
        c["t81"] = t81.decode(c["file"])[0]
        assert np.array_equal(c["t81"], c["coef"])
        c["want"] = port.decode(c["twin"])
        cases.append(c)
    assert sum(len(c["file"]) > 64 * 1024 for c in cases) >= 3 and sum(len(c["file"]) < 64 * 1024 for c in cases) >= 2
    files = [c["file"] for c in cases]
    for flags in (0, hjd.FLAG_HOST_SCAN, hjd.FLAG_NO_SELFSYNC):
        check(cases, decode(hjd, files, flags), flags)


@pytest.fixture(scope="module")
def nonsync(port):
    d = br.nonsync_case(2992, 3000, port=port)
    o = port.decode(d["file"])
    assert o["rc"] == 0 and np.array_equal(o["coef"], d["coef"])
    d["want"] = o
    return d


@pytest.mark.parametrize("ss_range", [32, 256])
def test_never_self_synchronises(hjd, nonsync, ss_range):
    """Every entry state of the speculative pass from sub-sequence 2 on is wrong (tests/test_baseline_random.py
    proves it in Python), so the rounds have to carry the correct state across every range: the decode is exact,
    the round limit is not hit (hjd_batch_get_status would fail), and it takes at most a round per range plus two."""
    f = nonsync["file"]
    n_subs = -(-(len(f) - br.scan_range(f)[0] - 2) // 128)
    with hjd.BatchDecoder(0) as d:
        d.set_selfsync_range(ss_range)
        d.upload([f])
        d.decode()
        st = d.status()
        assert st[0] == 0, st
        rounds = d.selfsync_rounds
        assert rounds <= -(-n_subs // ss_range) + 2, (rounds, n_subs)
        assert rounds > 2                                             # the chain did need the rounds
        assert np.array_equal(d.image_coefficients(0), nonsync["want"]["coef"])
        assert np.array_equal(d.rgb(0), nonsync["want"]["rgb"])


def test_never_self_synchronises_odd_blocks(hjd, port):
    """The same construction with 3-byte blocks, which do not divide a 1024-bit sub-sequence: exact."""
    d = br.nonsync_case(2992, 3000, block_bytes=3, port=port)
    o = port.decode(d["file"])
    assert o["rc"] == 0 and np.array_equal(o["coef"], d["coef"])
    got = decode(hjd, [d["file"]])
    assert got["status"][0] == 0
    assert np.array_equal(got["coef"][0], o["coef"]) and np.array_equal(got["rgb"][0], o["rgb"])
