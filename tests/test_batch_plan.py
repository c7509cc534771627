"""The batch planner (csrc/batch_plan.cpp) on the CPU: the index-limit guards and the invariants of the plan.

The planner is built here with g++ alone (tests/plan_driver.cpp prints the plan as JSON), which also shows it needs
no CUDA.  tests/test_gpu_scale.py refuses the same guard batches through hjd_batch_upload on a device and checks
that no device memory moves."""
from __future__ import annotations

import json
import os
import subprocess

import numpy as np
import pytest

from tests import multiscan_random as mr
from tests.test_gpu_scale import golden, with_scan_bytes, with_size
from tools.gen_jpegs import encode_jpeg, make_c5, synth_rgb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hls_jpeg_decoder_b200", "csrc")
SS_MIN_BYTES = 1024                      # HJD_SS_MIN_BYTES: shorter restart-free scans stay on kernel 1a


@pytest.fixture(scope="session")
def driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("plan") / "plan_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-pthread", "-o", exe, os.path.join(ROOT, "tests", "plan_driver.cpp"),
                           os.path.join(CSRC, "batch_plan.cpp"), os.path.join(CSRC, "jpeg_parse.cpp")])
    return exe


@pytest.fixture()
def plan(driver, tmp_path):
    def run(files, flags=0, overlap=1, chunk_images=0, chunked=True, repeat=1):
        paths = []
        for k, f in enumerate(files):
            paths.append(str(tmp_path / f"{k}.jpg"))
            with open(paths[-1], "wb") as fh:
                fh.write(f)
        out = subprocess.run([driver, str(flags), str(overlap), str(chunk_images), str(int(chunked)), str(repeat)] + paths,
                             check=True, capture_output=True, text=True).stdout
        for p in paths:
            os.remove(p)
        return json.loads(out)
    return run


# ------------------------------------------------------------------------------------------------
# guards: the same batches and messages as test_guard_blocks / test_guard_destuff_chunks
# ------------------------------------------------------------------------------------------------
def test_plan_guard_blocks(plan, hjd):
    big = with_size(golden("444_64x48_q85.jpg"), 16384, 16384)
    assert hjd.probe(big)[1].n_blocks == 12582912
    ok = plan([big], repeat=341)
    assert ok["rc"] == 0 and sum(im[15] for im in ok["images"]) == 341 * 12582912
    r = plan([big], repeat=342)
    assert r["rc"] == -1 and r["err"] == "batch exceeds 2^32 blocks", r


def test_plan_guard_destuff_chunks(plan):
    f = with_scan_bytes(golden("444_64x48_q85.jpg"), 2 ** 30)
    ok = plan([f], repeat=63)
    assert ok["rc"] == 0 and len(ok["ss"]) == 63
    r = plan([f], repeat=65)
    assert r["rc"] == -1 and "2^32 16-byte chunks" in r["err"], r


# ------------------------------------------------------------------------------------------------
# plan invariants
# ------------------------------------------------------------------------------------------------
def check_plan(p, files, flags, hjd):
    assert p["rc"] == 0, p
    imgs, chunks = p["images"], p["chunks"]
    n = len(files)
    assert len(imgs) == n
    # chunks are contiguous and cover every image
    assert chunks[0][0] == 0 and chunks[-1][1] == n
    for a, b in zip(chunks, chunks[1:]):
        assert a[1] == b[0] and a[0] < a[1]
    ss_of = {s[0]: k for k, s in enumerate(p["ss"])}

    # per-image geometry equals hjd.probe(buf, flags)
    for i, (f, im) in enumerate(zip(files, imgs)):
        st, o = hjd.probe(f, flags)
        assert im[0] == st, i
        if st != 0:
            continue
        assert im[1:11] == [o.width, o.height, o.ncomp, o.hf, o.vf, o.blocks_per_mcu, o.mcus_x, o.mcus_y,
                            o.restart_interval, im[10]], i
        assert im[12] == o.scan_bytes and im[15] == o.n_blocks, i
        want_intervals = im[17] if im[19] else (1 if i in ss_of else im[10])
        assert want_intervals == o.n_intervals, i

    work, segs = p["work"], p["segs"]
    sswork, sssegs, ss = p["sswork"], p["sssegs"], p["ss"]
    seen_iv = {}
    seen_spec, seen_sync = {}, {}
    seen_ms = {}
    mswork, scans = p["mswork"], p["scans"]
    for c in chunks:
        img0, img1, work0, work1, ss0, ss1, sw0, sw1, sf0, sf1, levels = c
        # kernel 1a: every interval in exactly one segment of this chunk's work range; CTAs of <= cap intervals, one table set
        for w in work[work0:work1]:
            first_seg, n_segs, n_iv, ts = w
            assert 0 < n_iv <= p["ent_threads"]
            tid = 0
            for s in segs[first_seg:first_seg + n_segs]:
                first, tid0, image, cnt = s
                assert img0 <= image < img1 and imgs[image][13] == ts and tid0 == tid
                tid += cnt
                for g in range(first, first + cnt):
                    assert imgs[image][11] <= g < imgs[image][11] + imgs[image][10]
                    seen_iv[g] = seen_iv.get(g, 0) + 1
            assert tid == n_iv
        # kernel 1b: every sub-sequence in one speculative and one sync segment of this chunk
        for lo, hi, seen, spec in ((sw0, sw1, seen_spec, True), (sf0, sf1, seen_sync, False)):
            for w in sswork[lo:hi]:
                first_seg, n_segs, n_subs, ts = w
                assert n_subs > 0 and (n_subs <= p["ss_threads"] if spec else 0 < n_segs <= p["ss_fix_warps"])
                tid = 0
                for s in sssegs[first_seg:first_seg + n_segs]:
                    k, first, tid0, cnt = s
                    assert ss0 <= k < ss1 and imgs[ss[k][0]][13] == ts
                    assert tid0 == (tid if spec else 0)
                    tid += cnt
                    for sub in range(first, first + cnt):
                        assert sub < ss[k][2]
                        seen[(k, sub)] = seen.get((k, sub), 0) + 1
                assert tid == n_subs
        # multi-scan: the chunk's items by non-decreasing level, the level ranges contiguous
        if levels:
            for (a, b), (c2, _) in zip(levels, levels[1:]):
                assert b == c2
            prev = -1
            for it in mswork[levels[0][0]:levels[-1][1]]:
                sc = scans[it[0]]
                assert img0 <= sc[0] < img1 and sc[1] >= prev and it[1] < sc[2]
                prev = sc[1]
                seen_ms[tuple(it)] = seen_ms.get(tuple(it), 0) + 1
            for a, b in levels:
                assert len({scans[it[0]][1] for it in mswork[a:b]}) == 1

    want_iv = sum(im[10] for im in imgs)
    assert len(seen_iv) == want_iv and set(seen_iv.values()) <= {1}
    want_subs = {(k, sub) for k, s in enumerate(ss) for sub in range(s[2])}
    assert set(seen_spec) == want_subs and set(seen_spec.values()) <= {1}
    assert set(seen_sync) == want_subs and set(seen_sync.values()) <= {1}
    want_ms = {(k, j) for k, s in enumerate(scans) for j in range(s[2])}
    assert set(seen_ms) == want_ms and set(seen_ms.values()) <= {1} and len(mswork) == len(want_ms)


def golden_files():
    d = os.path.join(ROOT, "tests", "golden")
    return [open(os.path.join(d, f), "rb").read() for f in sorted(os.listdir(d)) if f.endswith(".jpg")]


def restart_free_files():
    out = [encode_jpeg(synth_rgb(w, h, 7 + k), 85, sub, 0, gray=gray)
           for k, (w, h, sub, gray) in enumerate([(256, 192, "4:2:0", False), (200, 136, "4:4:4", False),
                                                  (320, 240, "4:2:0", True), (96, 80, "4:2:0", False)])]
    out.append(encode_jpeg(synth_rgb(128, 96, 3), 85, "4:2:0", 4))       # one restart-marker file among them
    return out


def multiscan_files(port):
    return [mr.random_case(s, w, h, sampling, port=port)["file"]
            for s, (w, h, sampling) in enumerate([(64, 48, "4:2:0"), (40, 40, "gray"), (72, 56, "4:4:4"),
                                                  (33, 17, "4:2:0"), (48, 64, "4:2:2")])]


CONFIGS = [dict(overlap=0, chunked=False), dict(overlap=1, chunked=True), dict(overlap=40, chunked=True),
           dict(overlap=1, chunked=True, chunk_images=3)]


@pytest.mark.parametrize("cfg", CONFIGS, ids=["overlap0", "overlap1", "overlap40", "chunk_images3"])
@pytest.mark.parametrize("case", ["golden", "c5", "restart_free", "multiscan"])
def test_plan_invariants(plan, hjd, port, case, cfg):
    flags = 0
    if case == "golden":
        files = golden_files()
    elif case == "c5":
        files = [make_c5(i) for i in range(24)] + [make_c5(i, restart=False) for i in range(24, 32)]
    elif case == "restart_free":
        files = restart_free_files()
        assert all(len(f) > SS_MIN_BYTES + 1024 for f in files)
    else:
        flags = hjd.FLAG_MULTI_SCAN
        files = multiscan_files(port) + [golden_files()[0]]
    p = plan(files, flags=flags, **cfg)
    check_plan(p, files, flags, hjd)
    if case == "restart_free":
        assert len(p["ss"]) == 4 and len(p["sswork"]) > 0
    if case == "multiscan":
        assert len(p["mswork"]) > 0 and sum(im[19] for im in p["images"]) == 5
    if cfg.get("overlap") == 40:
        assert len(p["chunks"]) > 1
