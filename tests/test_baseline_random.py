"""Random baseline files on the host (no GPU): the writer's random tables, selectors, restart layouts, fill bytes
and wrapping DC walks round-trip through the T.81 restatement (tests/t81_decode.py), the oracle agrees wherever
it can decode the file, and the batch that tests/test_gpu_baseline_random.py decodes reaches what it claims to.
Also: the non-synchronising stream of that test has the chain of wrong speculative entry states it claims."""
from __future__ import annotations

import numpy as np
import pytest

from tests import baseline_random as br
from tests import t81_decode as t81

N_EXTRA = 60          # random cases beyond the batch: random restart layouts, fill and walks


def oracle_coef(port, c):
    """The oracle's entropy decode, with its 16-bit DC switch where a DC table has a 16-bit code."""
    port.set_dc16(c["stats"]["dc16"])
    try:
        return port.decode(c["file"], entropy_only=True)
    finally:
        port.set_dc16(False)


@pytest.fixture(scope="module")
def cases(port):
    out = [br.random_case(**br.batch_params(i), port=port) for i in range(br.N_BATCH)]
    for seed in range(N_EXTRA):
        w, h = br.SIZES[seed % len(br.SIZES)]
        out.append(br.random_case(seed, w, h, br.SAMPLINGS[seed % len(br.SAMPLINGS)], port=port))
    return out


def test_t81_and_oracle_agree(port, cases):
    refused = 0
    for i, c in enumerate(cases):
        coef, g, _ = t81.decode(c["file"])
        assert np.array_equal(coef, c["coef"]), i                      # the DC reduced mod 2^16 where it wraps
        assert all(g[k] == c["geometry"][k] for k in ("width", "height", "ncomp", "hf", "vf", "mcus_x", "mcus_y"))
        o = oracle_coef(port, c)
        if c["stats"]["fill_before_rst"]:
            # the reference pairs RSTn with the byte after the interval's data (HJDO_ERR_RESTART): T.81 B.1.1.2 is
            # the only reference for these files
            assert o["rc"] == -5, (i, o["rc"])
            refused += 1
            continue
        assert o["rc"] == 0, (i, o["rc"])
        assert np.array_equal(o["coef"], c["coef"]), i
        tw = port.decode(c["twin"], entropy_only=True)
        assert tw["rc"] == 0 and np.array_equal(tw["coef"], c["coef"]), i
    assert refused >= 5


def test_batch_coverage(cases):
    """What the GPU batch has to reach, asserted rather than hoped for."""
    batch = cases[:br.N_BATCH]
    lengths, phases, fill, zrl = set(), set(), 0, 0
    wrapped, dris, kinds = set(), set(), set()
    for i, c in enumerate(batch):
        _, _, cov = t81.decode(c["file"])
        lengths |= cov["code_lengths"]["seq_dc"] | cov["code_lengths"]["seq_ac"]
        fill += cov["fill_bytes"]
        zrl += cov["seq_zrl"]
        phases |= c["stats"]["ff00"]
        if c["stats"]["wrapped"]:
            wrapped.add(c["geometry"]["ncomp"] == 1 and "gray" or (c["geometry"]["hf"], c["geometry"]["vf"]))
        n, d = c["stats"]["n_mcus"], c["dri"]
        dris.add(d if isinstance(d, str) else {n - 1: "m-1", n: "m", n + 5: "m+5"}.get(d, d))
        kinds |= set(c["stats"]["kinds"].values())
    assert lengths == set(range(1, 17)), sorted(lengths)
    assert fill > 0 and zrl > 0
    assert {"gray", (2, 2), (1, 1)} <= wrapped, wrapped                 # gray, 4:2:0 and 4:4:4
    assert phases == set(range(16))                                    # FF 00 at every phase; FF last of a chunk
    assert {0, "dri0", 1, "m-1", "m", "m+5", 65535} <= dris, dris
    assert {"flat", "long", "mixed", "single", "shared"} <= kinds, kinds
    assert sum(c["stats"]["sof1"] for c in batch) >= 8
    assert sum(c["stats"]["decoy"] for c in batch) >= 4
    assert sum(c["stats"]["fill_before_rst"] for c in batch) >= 4
    assert sum(c["fill"] > 0 and c["stats"]["n_intervals"] == 1 for c in batch) >= 4      # fill before EOI only
    n_free = sum(c["stats"]["n_intervals"] == 1 for c in batch)
    assert 16 <= n_free <= br.N_BATCH - 16                             # restart-free and restart cases mixed
    # several restart-free images with different table sets: kernel 1b's sync kernel reloads its tables
    assert len({repr(sorted(c["tables"].items())) for c in batch if c["stats"]["n_intervals"] == 1}) >= 8


def test_writer_defaults_unchanged(port):
    """The new keyword arguments of jpeg_writer.rewrite default to the old output, byte for byte."""
    from tests import jpeg_writer as jw
    from tests import multiscan_random as mr
    tmpl = mr.template(40, 24, "4:2:0")
    o = port.decode(tmpl, entropy_only=True)
    for ri in (0, 3):
        a = jw.rewrite(tmpl, o["coef"], o["geometry"], restart_interval=ri)
        b = jw.rewrite(tmpl, o["coef"], o["geometry"], restart_interval=ri, selectors=None, fill=0, dc_mod16=False,
                       decoy=None, dht_order=None, sof_marker=None, dri_segment=False, zrl_tail=())
        assert a == b and np.array_equal(t81.decode(a)[0], o["coef"])


def test_nonsync_chain(port):
    """The non-synchronising stream (the GPU test's 2992x3000 4:4:4 image): every 128-byte sub-sequence boundary is a
    block start, the block-in-MCU index there is 1 from sub-sequence 1 on, and kernel 1b's speculative pass (thread li
    decodes sub-sequence li - 1 from (bit (li - 1) * 1024, k = 0, block 0)) enters every sub-sequence from 2 on with
    the wrong index; its states are consistent with each other everywhere except between sub-sequences 1 and 2, so
    only the synchronisation rounds, one sub-sequence after another, can correct them."""
    d = br.nonsync_case(2992, 3000, port=port)
    o = port.decode(d["file"], entropy_only=True)
    assert o["rc"] == 0 and np.array_equal(o["coef"], d["coef"])
    a, e = br.scan_range(d["file"])
    data = d["file"][a:e]
    assert 0xFF not in data                                            # no stuffing: de-stuffed == scan
    x, ex = br.spec_states(data)
    truth = br.true_states(d["lengths"])
    n = len(x)
    assert 4096 <= n <= 16384
    assert all(t is not None for t in truth)                           # a block starts at every boundary
    assert all(truth[li][2] == 1 for li in range(1, n))
    assert x[0] == truth[0] and x[1] == truth[1]
    assert all(x[li] != truth[li] for li in range(2, n))
    assert all(x[li][:2] == truth[li][:2] for li in range(n))          # wrong only in the block-in-MCU index
    assert [li for li in range(1, n) if ex[li - 1] != x[li]] == [2]
    # a small one decodes under T.81 to the coefficients it was built from; so does the 3-byte-block variant
    for bb in (None, 3):
        s = br.nonsync_case(120, 64, block_bytes=bb, port=port)
        assert np.array_equal(t81.decode(s["file"])[0], s["coef"])
