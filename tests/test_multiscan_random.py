"""Random legal multi-scan files on the host (no GPU): the reference decoder tests/t81_decode.py pinned against the
oracle, the writer's random scripts, tables and fill bytes round-tripped through it and through Pillow, and the
host parse (probe, scans, work items, dependency levels) of every such file."""
from __future__ import annotations

import io

import numpy as np
import pytest
from PIL import Image

from tests import multiscan_random as mr
from tests import multiscan_writer as mw
from tests import t81_decode as t81
from tests.multiscan_writer import coded_mask
from tests.test_multiscan_host import PAIRS, WRITER_CASES, writer_files

SIZES = [(1, 1), (17, 9), (37, 53), (61, 35), (8, 8), (24, 40), (64, 48), (33, 17)]
N_SEEDS = 200


def case_params(seed: int):
    """(width, height, sampling, sequential, complete) of random case `seed`: small odd sizes, every 25th 333x217;
    two colour cases in seven sequential; every other one coded down to Al 0 everywhere."""
    sampling = mr.SAMPLINGS[seed % len(mr.SAMPLINGS)]
    w, h = (333, 217) if seed % 25 == 7 else SIZES[(seed // 5) % len(SIZES)]
    return w, h, sampling, seed % 7 in (3, 6) and sampling != "gray", seed % 2 == 0


def pillow_comparable(script, ncomp: int) -> bool:
    """libjpeg smooths the blocks of a progressive image whose DC or first AC coefficients are not all known to
    Al 0 (block smoothing, jdcoefct.c), so Pillow's pixels equal the twin's only when every component's coefficients
    0..9 end at Al 0."""
    final = {}
    for comps, ss, se, ah, al in script:
        for c in comps:
            for k in range(ss, se + 1):
                final[(c, k)] = al
    return all(final.get((c, k)) == 0 for c in range(ncomp) for k in range(10))


def level_invariant(scans):
    """Scans that share a (component, coefficient) position have strictly increasing levels in file order; scans on
    one level share no position."""
    pos = [{(c, k) for c in s["comp"] for k in range(s["ss"], s["se"] + 1)} for s in scans]
    for i in range(len(scans)):
        for j in range(i + 1, len(scans)):
            if pos[i] & pos[j]:
                assert scans[i]["level"] < scans[j]["level"], (i, j)
            if scans[i]["level"] == scans[j]["level"]:
                assert not pos[i] & pos[j], (i, j)


def check_host_parse(hjd, f, script, restarts, geometry):
    st, info = hjd.probe(f, hjd.FLAG_MULTI_SCAN)
    assert st == 0
    sc = hjd.scans(f)
    assert [(tuple(s["comp"]), s["ss"], s["se"], s["ah"], s["al"]) for s in sc] == [tuple(s) for s in script]
    assert [s["restart_interval"] for s in sc] == list(restarts)
    want = sum(-(-mr.scan_grid(geometry, comps) // ri) if ri else 1 for (comps, *_), ri in zip(script, restarts))
    assert info.n_intervals == want
    level_invariant(sc)
    return sc


# C1: the reference decoder equals the oracle on libjpeg-turbo's files and the writer's existing variants

@pytest.mark.parametrize("name", sorted(PAIRS))
def test_reference_decoder_on_libjpeg_files(port, name):
    prog, twin = PAIRS[name]()
    o = port.decode(twin, entropy_only=True)
    coef, g, cov = t81.decode(prog)
    m = coded_mask(o["geometry"])
    assert np.array_equal(coef[m], o["coef"][m])
    assert all(g[k] == o["geometry"][k] for k in ("width", "height", "ncomp", "hf", "vf", "mcus_x", "mcus_y"))


def test_reference_decoder_on_twin_cases(port):
    from tests.test_gpu_multiscan import TWIN_CASES
    for name, make in TWIN_CASES.items():
        prog, twin = make()
        o = port.decode(twin, entropy_only=True)
        m = coded_mask(o["geometry"])
        assert np.array_equal(t81.decode(prog)[0][m], o["coef"][m]), name


@pytest.mark.parametrize("case", WRITER_CASES)
def test_reference_decoder_on_writer_files(port, case):
    from tests.cases import small_cases
    f = small_cases()[case]
    o = port.decode(f, entropy_only=True)
    m = coded_mask(o["geometry"])
    for name, b in writer_files(f, port).items():
        assert np.array_equal(t81.decode(b)[0][m], o["coef"][m]), name


# C2 and C3: random scripts, tables and coefficients

def test_random_files_round_trip(hjd, port):
    pooled = dict(code_lengths={}, eobn={"ac_first": set(), "ac_refine": set()}, comps=set(), fill=0, al={})
    compared = seq_ac = seq_zrl = 0
    cases = [(seed, mr.random_case(seed, *case_params(seed)[:3], sequential=case_params(seed)[3],
                                   complete=case_params(seed)[4], port=port)) for seed in range(N_SEEDS)]
    # plus one 1024x1040 gray image (16,640 blocks) with runs of empty blocks of every length 2^n up to 8192: EOBn
    # up to 13 in both AC kinds
    tmpl = mr.template(1024, 1040, "gray")
    g = port.decode(tmpl, entropy_only=True)["geometry"]
    ladder = mr.eob_ladder(g, 5)
    from tests.jpeg_writer import blocks_to_jpeg
    twin = blocks_to_jpeg(tmpl, ladder, g, {0: np.ones(64, int)})
    cases.append(("ladder", dict(file=mw.write_multiscan(twin, ladder, g, mw.DEFAULT_SCRIPT_GRAY, tables="mixed"),
                                 twin=twin, script=mw.DEFAULT_SCRIPT_GRAY, restarts=[0] * 6, expected=ladder,
                                 geometry=g)))
    for seed, c in cases:
        g = c["geometry"]
        coef, g2, cov = t81.decode(c["file"])
        assert np.array_equal(coef, c["expected"]), seed
        if seed != "ladder":
            assert np.array_equal(c["expected"], mw.expected_after(c["coef"], g["ncomp"], g, c["script"],
                                                                   len(c["script"])))
        if pillow_comparable(c["script"], g["ncomp"]):
            got = np.asarray(Image.open(io.BytesIO(c["file"])).convert("RGB"))
            want = np.asarray(Image.open(io.BytesIO(c["twin"])).convert("RGB"))
            assert np.array_equal(got, want), seed
            compared += 1
        sc = check_host_parse(hjd, c["file"], c["script"], c["restarts"], g)
        # beyond the invariant: the host puts every scan on the earliest level it may take, so an image needs no
        # more launches than its longest dependency chain
        assert max(s["level"] for s in sc) + 1 == cov["levels"], seed
        if seed != "ladder" and case_params(seed)[3]:          # a sequential file
            seq_ac = max(seq_ac, cov["seq_ac_nonzero"])
            seq_zrl += cov["seq_zrl"]
        for k, v in cov["code_lengths"].items():
            pooled["code_lengths"].setdefault(k, set()).update(v)
        for k in ("ac_first", "ac_refine"):
            pooled["eobn"][k] |= cov["eobn"][k]
        for k, v in cov["al"].items():
            pooled["al"].setdefault(k, set()).update(v)
        pooled["comps"] |= set(cov["scan_comps"])
        pooled["fill"] += cov["fill_bytes"]
    assert compared >= N_SEEDS // 3
    assert seq_ac > 1000 and seq_zrl > 0             # sequential scans code whole blocks, not just their DC
    for kind in ("seq_dc", "seq_ac", "dc_first", "ac_first", "ac_refine"):
        assert pooled["code_lengths"][kind] == set(range(1, 17)), (kind, pooled["code_lengths"][kind])
    for kind in ("ac_first", "ac_refine"):
        assert set(range(14)) <= pooled["eobn"][kind], (kind, pooled["eobn"][kind])
    assert {(1, 2), (0, 2)} <= pooled["comps"]
    assert pooled["fill"] > 0
    assert 13 in pooled["al"]["dc_first"] and 13 in pooled["al"]["ac_first"]


def test_long_and_mixed_tables():
    """The random tables are canonical codes of the right symbols that never assign the all-ones code; "long" ones
    hold no code under 11 bits, "mixed" ones one of each length 11..16 from six symbols on.  (The host builds
    every table of every random file when test_random_files_round_trip probes it.)"""
    rng = np.random.default_rng(1)
    for n in (1, 2, 5, 6, 7, 40, 162, 256):
        for _ in range(20):
            symbols = list(range(n))
            for make, lo in ((mw.long_table, 11), (mw.mixed_table, 1)):
                bits, vals = make(symbols, rng)
                assert sum(bits) == n and sorted(vals) == symbols
                assert sum(b << (16 - L) for L, b in enumerate(bits, 1)) < 1 << 16          # never all ones
                assert not any(bits[:lo - 1])
                if make is mw.mixed_table and n >= 6:
                    assert all(bits[L - 1] for L in range(11, 17))
