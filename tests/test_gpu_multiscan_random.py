"""HJD_FLAG_MULTI_SCAN on random legal scripts, long and mixed Huffman codes, extreme coefficients, maximal EOB runs
and a 256-scan file: the GPU slab equals the reference decoder (tests/t81_decode.py) and the coefficients the script
codes, bit for bit, and RGB equals the oracle's decode of the baseline twin."""
from __future__ import annotations

import numpy as np
import pytest

from tests import multiscan_random as mr
from tests import multiscan_writer as mw
from tests import t81_decode as t81
from tests.jpeg_writer import blocks_to_jpeg

pytestmark = pytest.mark.gpu

N_BATCH = 48
SIZES = [(1, 1), (17, 9), (37, 53), (61, 35), (64, 48), (120, 88), (333, 217)]


def decode(hjd, files, flags=0, dec=None):
    """(status, [dict(coef, rgb, scans, info)]) of one batch; `dec`: an open handle to reuse."""
    own = dec is None
    if own:
        dec = hjd.BatchDecoder(0, flags | hjd.FLAG_MULTI_SCAN)
    try:
        dec.upload(files)
        dec.decode()
        st = dec.status()
        coef = dec.coefficients()
        out = [dict(coef=dec.image_coefficients(i, coef).copy(), rgb=dec.rgb(i).copy(), scans=dec.num_scans(i),
                    info=dec.info(i)) for i in range(len(files))]
    finally:
        if own:
            dec.close()
    return st, out


@pytest.fixture(scope="module")
def batch(port):
    cases = []
    for seed in range(N_BATCH):
        sampling = mr.SAMPLINGS[seed % len(mr.SAMPLINGS)]
        w, h = SIZES[seed % len(SIZES)]
        c = mr.random_case(1000 + seed, w, h, sampling, sequential=seed % 8 == 5 and sampling != "gray",
                           complete=seed % 3 == 0, port=port)
        c["t81"], _, c["cov"] = t81.decode(c["file"])
        cases.append(c)
    return cases


def uncoded(script, ncomp: int) -> bool:
    """Whether some (component, coefficient) position is coded by no scan of `script`."""
    coded = {(c, k) for comps, ss, se, _, _ in script for c in comps for k in range(ss, se + 1)}
    return len(coded) < 64 * ncomp


def test_random_batch(hjd, port, batch):
    # what the batch has to reach: interleavings that do not start at component 0, positions no scan codes (so that
    # stale slab contents would show), and sequential scans with AC data
    assert {(1, 2), (0, 2)} <= {t for c in batch for t in c["cov"]["scan_comps"]}
    assert sum(uncoded(c["script"], c["geometry"]["ncomp"]) for c in batch) >= 5
    assert max(c["cov"]["seq_ac_nonzero"] for c in batch) > 0
    files = [c["file"] for c in batch]
    st, out = decode(hjd, files)
    assert (st == 0).all(), st
    for i, (c, r) in enumerate(zip(batch, out)):
        assert r["scans"] == len(c["script"]), i
        assert np.array_equal(r["coef"], c["t81"]), i
        assert np.array_equal(r["coef"], c["expected"]), i
        assert np.array_equal(r["rgb"], port.decode(c["twin"])["rgb"]), i
    st_r, out_r = decode(hjd, files[::-1])
    assert (st_r == 0).all()
    for a, b in zip(out, out_r[::-1]):
        assert np.array_equal(a["coef"], b["coef"]) and np.array_equal(a["rgb"], b["rgb"])
    # the same handle after a batch of noise baseline images: blocks no scan codes are 0, not what the slab held
    rng = np.random.default_rng(7)
    from tools.gen_jpegs import encode_jpeg
    noise = [encode_jpeg(rng.integers(0, 256, (217, 333, 3), dtype=np.uint8), 100, "4:4:4") for _ in range(len(files))]
    with hjd.BatchDecoder(0, hjd.FLAG_MULTI_SCAN) as dec:
        st_n, _ = decode(hjd, noise, dec=dec)
        assert (st_n == 0).all()
        st2, out2 = decode(hjd, files, dec=dec)
    assert (st2 == 0).all()
    for i, (a, b) in enumerate(zip(out, out2)):
        assert np.array_equal(a["coef"], b["coef"]) and np.array_equal(a["rgb"], b["rgb"]), i


DEEP_GRAY = [((0,), 0, 0, 0, 0), ((0,), 1, 5, 0, 3), ((0,), 6, 63, 0, 3), ((0,), 1, 63, 3, 2), ((0,), 1, 63, 2, 1),
             ((0,), 1, 63, 1, 0)]


@pytest.mark.timeout(300)
def test_maximal_eob_runs(hjd, port):
    cases = []
    for sampling, w, h, rungs in (("gray", 1536, 1536, True), ("4:2:0", 2048, 1024, False)):
        tmpl = mr.template(w, h, sampling)
        g = port.decode(tmpl, entropy_only=True)["geometry"]
        coef = mr.eob_ladder(g, 3, corrections=40, rungs=rungs)
        quant = {0: np.ones(64, int), 1: np.ones(64, int)} if g["ncomp"] == 3 else {0: np.ones(64, int)}
        twin = blocks_to_jpeg(tmpl, coef, g, quant)
        default = mw.DEFAULT_SCRIPT_GRAY if sampling == "gray" else mw.DEFAULT_SCRIPT_COLOR
        deep = DEEP_GRAY if sampling == "gray" else [((0, 1, 2), *s[1:]) if s[1] == 0 else s for s in DEEP_GRAY] + \
            [((c,), 1, 63, 0, 0) for c in (1, 2)]
        for script in (default, deep):
            for dri in (0, 1000):
                f = mw.write_multiscan(twin, coef, g, script, restarts=[dri] * len(script), tables="mixed")
                cases.append((f, twin, script, coef, g))
    st, out = decode(hjd, [c[0] for c in cases])
    assert (st == 0).all(), st
    for i, ((f, twin, script, coef, g), r) in enumerate(zip(cases, out)):
        assert r["scans"] == len(script)
        want, _, cov = t81.decode(f)
        assert np.array_equal(want, mw.expected_after(coef, g["ncomp"], g, script, len(script))), i
        assert np.array_equal(r["coef"], want), i
        assert np.array_equal(r["rgb"], port.decode(twin)["rgb"]), i
        if i % 2 == 0:                                    # DRI 0: the runs reach EOB14
            assert 14 in cov["eobn"]["ac_first"] and 14 in cov["eobn"]["ac_refine"], (i, cov["eobn"])
            assert cov["max_eob_corrections"] >= 900, (i, cov["max_eob_corrections"])


def scan_cap_script():
    """256 scans: DC from Al 13 refined to 0, then single-coefficient AC bands from Al 13 refined towards 0."""
    script = [((0,), 0, 0, 0, 13)] + [((0,), 0, 0, al + 1, al) for al in range(12, -1, -1)]
    k = 1
    while len(script) < 256:
        script.append(((0,), k, k, 0, 13))
        for al in range(12, -1, -1):
            script.append(((0,), k, k, al + 1, al))
        k += 1
    return script[:256]


def test_256_scans(hjd, port):
    tmpl = mr.template(48, 40, "gray")
    g = port.decode(tmpl, entropy_only=True)["geometry"]
    coef = mr.random_coefficients(np.random.default_rng(11), g)
    script = scan_cap_script()
    want = mw.expected_after(coef, 1, g, script, len(script))
    twin = blocks_to_jpeg(tmpl, want, g, {0: np.full(64, 2)})
    f = mw.write_multiscan(twin, want, g, script, restarts=[(k % 4) * 3 for k in range(256)], tables="mixed")
    ref, _, cov = t81.decode(f)
    assert cov["levels"] >= 14
    sc = hjd.scans(f)
    # the host puts every scan on the earliest level it may take: as many launches as the longest dependency chain
    assert len(sc) == 256 and max(s["level"] for s in sc) + 1 == cov["levels"]
    st, out = decode(hjd, [f, twin, f])
    assert (st == 0).all(), st
    for r in (out[0], out[2]):
        assert r["scans"] == 256
        assert np.array_equal(r["coef"], want) and np.array_equal(ref, want)
        assert np.array_equal(r["rgb"], port.decode(twin)["rgb"])


def test_cut_after_each_scan(hjd, port):
    files, want = [], []
    for seed, sampling in ((21, "4:2:0"), (22, "4:4:4"), (23, "gray")):
        c = mr.random_case(seed, 37, 29, sampling, max_scans=40, port=port)
        for k in range(1, len(c["script"]) + 1):
            f = mw.write_multiscan(c["twin"], c["expected"], c["geometry"], c["script"], restarts=c["restarts"],
                                   tables=c["tables"], fill=c["fill"], seed=seed, truncate_after=k)
            files.append(f)
            e = mw.expected_after(c["expected"], c["geometry"]["ncomp"], c["geometry"], c["script"], k)
            assert np.array_equal(t81.decode(f)[0], e), (seed, k)
            want.append((k, e))
    st, out = decode(hjd, files)
    assert (st == 0).all(), st
    for (k, e), r in zip(want, out):
        assert r["scans"] == k
        assert np.array_equal(r["coef"], e), k


def test_scaled_output(hjd, port, batch):
    from tests import scaled_port
    files = [c["file"] for c in batch]
    st, out = decode(hjd, files, hjd.FLAG_SCALE_1_8)
    assert (st == 0).all(), st
    for i, (c, r) in enumerate(zip(batch, out)):
        dc = [s for s, ri in zip(c["script"], c["restarts"]) if s[1] == 0]
        items = sum(-(-mr.scan_grid(c["geometry"], s[0]) // ri) if ri else 1
                    for s, ri in zip(c["script"], c["restarts"]) if s[1] == 0)
        assert r["scans"] == len(dc), i
        assert r["info"].n_intervals == items, i
        assert np.array_equal(r["coef"], mw.expected_after(c["expected"], c["geometry"]["ncomp"], c["geometry"], dc,
                                                           len(dc))), i
        assert np.array_equal(r["rgb"], scaled_port.decode_scaled(c["twin"], 3)["rgb"]), i
    st, out = decode(hjd, files, hjd.FLAG_SCALE_1_2)
    assert (st == 0).all(), st
    for i, (c, r) in enumerate(zip(batch, out)):
        assert r["scans"] == len(c["script"])
        assert np.array_equal(r["coef"], c["t81"]), i
        assert np.array_equal(r["rgb"], scaled_port.decode_scaled(c["twin"], 1)["rgb"]), i


def test_chunks_and_devices(hjd, port, batch):
    files = [c["file"] for c in batch]
    want = [port.decode(c["twin"])["rgb"] for c in batch]
    arena = hjd.PinnedArena(files)
    try:
        with hjd.BatchDecoder(0, hjd.FLAG_MULTI_SCAN) as dec:
            dec.set_overlap(1)
            cap = int(hjd.lib().hjd_out_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n, hjd.FLAG_MULTI_SCAN))
            out = np.zeros(cap, np.uint8)
            offs, st = dec.decode_host(arena, out.ctypes.data, cap, 3)
            assert (st == 0).all(), st
            for i, w in enumerate(want):
                h, wd = w.shape[:2]
                assert np.array_equal(out[offs[i]:offs[i] + h * wd * 3].reshape(h, wd, 3), w), i
        with hjd.MultiDecoder([0, 0], flags=hjd.FLAG_MULTI_SCAN) as md:
            cap = md.out_slab_bytes(arena)
            out = np.zeros(cap, np.uint8)
            offs, st = md.decode_host(arena, out.ctypes.data, cap)
            assert (st == 0).all(), st
            for i, w in enumerate(want):
                h, wd = w.shape[:2]
                assert np.array_equal(out[offs[i]:offs[i] + h * wd * 3].reshape(h, wd, 3), w), i
    finally:
        arena.close()
