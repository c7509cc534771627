"""CPU checks of the committed adversarial IDCT block set (tests/golden/idct_edges.npz, tools/make_idct_edges.py):
every label is re-derived from the emulations of the two kernels' fast tiers and the reference's float order, so the
set cannot silently stop reaching the boundaries it was built for; and the premise of the tensor-core kernel's error
window -- its FP16 estimate of A -- is checked in the kernel's own order of operations."""
import os

import numpy as np
import pytest

from tools import make_idct_edges as E

NPZ = os.path.join(os.path.dirname(__file__), "golden", "idct_edges.npz")

MIN_COUNTS = {"tc_fast_wrong": 20, "cc_fast_wrong": 20, "cc_short_fast_wrong": 8, "near_integer": 8,
              "near_sat_m129": 2, "near_sat_m128": 2, "near_sat_127": 2, "near_sat_128": 2, "row_flagged": 16,
              "ac_range_in": 6, "ac_range_out": 6, "dq_in": 3, "dq_out": 4, "dc_in": 3, "dc_out": 4,
              "a_below": 3, "a_above": 3, "a_fp16_worst": 2, "dc_only": 3, "dc_only_wide": 3,
              "dc_plus_1": 2, "dc_plus_63": 2, "last_20": 8, "last_21": 8}


@pytest.fixture(scope="module")
def edges():
    d = np.load(NPZ)
    T = E.Tables()
    coef, qidx, label = d["coef"], d["qidx"].astype(np.int64), d["label"]
    assert np.array_equal(d["quant"], E.QUANT)
    return T, coef, qidx, label, E.classify(T, coef, qidx)


def test_numpy_reference_is_the_oracle(edges):
    """The numpy float order the labels rest on gives the oracle's bytes (hjdo_decode_single_block) for every block."""
    from oracle import port
    T, coef, qidx, label, K = edges
    for i in range(coef.shape[0]):
        want = port.decode_single_block(coef[i], E.QUANT[qidx[i]].astype(np.float32)).ravel()
        assert np.array_equal(K["ref"][i], want), (i, label[i])


def test_every_label_holds(edges):
    T, coef, qidx, label, K = edges
    tc = K["tc"]
    fast = K["tc_fast"]
    rowflags = tc["flagged"].reshape(-1, 8, 8).sum(axis=2).max(axis=1)
    holds = {
        "tc_fast_wrong": K["tc_wrong"],
        "cc_fast_wrong": K["cc_wrong"] & (K["last"] > 20),
        "cc_short_fast_wrong": K["cc_wrong"] & (K["last"] <= 20),
        "near_integer": K["near_any"],
        "near_sat_m129": K["near_sat"][-129], "near_sat_m128": K["near_sat"][-128],
        "near_sat_127": K["near_sat"][127], "near_sat_128": K["near_sat"][128],
        "row_flagged": (rowflags == 8) & fast,
        "ac_range_in": fast, "ac_range_out": tc["all_exact"] & ~tc["dc_wide"],
        "dq_in": fast, "dq_out": tc["all_exact"],
        "dc_in": fast, "dc_out": tc["all_exact"] & tc["dc_wide"],
        "a_below": fast & (tc["a_tot"] < 4000), "a_above": tc["all_exact"] & ~tc["dc_wide"] & (tc["a_tot"] >= 4000),
        "a_fp16_worst": fast & (tc["acc"].astype(np.float32).max(axis=1) > 2048),
        "dc_only": tc["dc_only"], "dc_only_wide": ~tc["dc_only"] & tc["all_exact"] & (K["last"] == 0),
        "dc_plus_1": ~tc["dc_only"] & (K["last"] == 1), "dc_plus_63": ~tc["dc_only"] & (K["last"] == 63),
        "last_20": K["last"] == 20, "last_21": K["last"] == 21,
    }
    names, counts = np.unique(label, return_counts=True)
    assert set(names) == set(holds), set(names) ^ set(holds)
    for name, k in zip(names, counts):
        bad = np.nonzero((label == name) & ~holds[name])[0]
        assert len(bad) == 0, (name, bad)
        assert k >= MIN_COUNTS[name], (name, k)
    # the neighbours of a precondition differ in one coefficient: the pairs really straddle it
    for lo, hi in (("a_below", "a_above"),):
        a, b = coef[label == lo].astype(np.int64), coef[label == hi].astype(np.int64)
        assert ((a != b).sum(axis=1) == 1).all() and (np.abs(a - b).sum(axis=1) == 1).all()
    assert (tc["a_tot"][label == "a_below"] > 3950).all()


def test_both_tiers_are_right_where_they_accept(edges):
    """What each kernel keeps from its fast tier is the reference's byte; what the shortcut stores is too.  With the
    error windows at zero both fast tiers are wrong on the blocks labelled so."""
    T, coef, qidx, label, K = edges
    ref = K["ref"]
    for tier in (K["tc"], K["cc"]):
        kept = ~tier["flagged"]
        assert (tier["fast"][kept] == ref[kept]).all()
    dc = K["tc"]["dc_only"]
    assert (K["tc"]["dc_byte"][dc, None] == ref[dc]).all()
    q = E.QUANT[qidx]
    zero = E.tc_fast_tier(T, coef, q, window_units=0.0)
    wrong = ((zero["fast"] != ref) & ~zero["flagged"]).any(axis=1)
    assert wrong[label == "tc_fast_wrong"].all()


def test_fp16_estimate_of_a_bounds_the_error_window():
    """mcu_tc.cuh:383-421: A is summed in four FP16 accumulators (zig-zag position mod 4) with C(u)C(v) rounded up,
    added pairwise in FP16, then in FP32 with 0.5 |DC|, times 1.02.  Wherever that estimate admits a block
    (a_tot < 4000), the window it gives must be at least 18 units of the true A, and sum |v| < 8192 (the bound the
    fast tier's exactness rests on).  Dense random blocks, the committed set, and FP16 sums pushed past 2048."""
    T = E.Tables()
    rng = np.random.default_rng(7)
    blocks = [E._dense(rng, 20000, budget=int(b)) for b in (1500, 3000, 3600, 4200)]
    d = np.load(NPZ)
    blocks.append(d["coef"][d["qidx"] == 0].astype(np.int64))
    blocks.append(d["coef"][d["label"] == "a_fp16_worst"].astype(np.int64))
    coef = np.concatenate(blocks)
    q = np.ones((coef.shape[0], 64), dtype=np.uint8)
    tc = E.tc_fast_tier(T, coef, q)
    _, A = E.reference(T, coef, q)
    fast = ~tc["all_exact"] & ~tc["dc_only"]
    assert fast.sum() > 20000
    win_units = tc["win"][fast].astype(np.float64) / (A[fast] * E.UNIT)
    assert win_units.min() >= 18.0, win_units.min()
    assert (np.abs(coef[fast]).sum(axis=1) < 8192).all()
    ratio = A[fast] / (tc["a_tot"][fast].astype(np.float64) / 1.02)      # true A over the FP16 estimate
    assert ratio.max() < 1.016, ratio.max()                             # DESIGN 4.5: low by < 1.6 %
    print(f"worst true-A / FP16-estimate ratio: {ratio.max():.5f} (window >= {win_units.min():.2f} units)")


def test_generator_reproduces_the_committed_set():
    """tools/make_idct_edges.py is seeded: it writes this set again (the arrays; the file itself byte for byte with
    the same numpy and zlib)."""
    d = E.build()
    c = np.load(NPZ)
    assert sorted(d) == sorted(c.files)
    for k in d:
        assert np.array_equal(d[k], c[k]), k


def test_writer_places_blocks_and_tables():
    """jpeg_writer: a re-emitted scan decodes to the coefficients it was given, with the file's own quantisation
    tables or with the ones given per component (the oracle reads them back through its planes)."""
    from oracle import port
    from tests import cases
    from tests import jpeg_writer as jw
    src = cases.small_cases()["420_64x48_q85"]
    o = port.decode(src)
    same = port.decode(jw.rewrite(src, o["coef"], o["geometry"], restart_interval=3))
    assert same["rc"] == 0 and np.array_equal(same["coef"], o["coef"]) and np.array_equal(same["rgb"], o["rgb"])
    g = o["geometry"]
    blocks = np.zeros_like(o["coef"])
    i = jw.block_index(g, 3, mcu=5, comp=1)
    blocks[i, [0, 1, 20]] = [-300, 17, -4]
    qs = [E.QUANT[0], E.QUANT[1], E.QUANT[3]]
    f = jw.blocks_to_jpeg(src, blocks, g, {0: qs[0], 1: qs[1], 2: qs[2]}, tq=[0, 1, 2])
    d = port.decode(f)
    assert d["rc"] == 0 and np.array_equal(d["coef"], blocks)
    my, mx = divmod(5, g["mcus_x"])
    cb = d["planes"][1][8 * my:8 * my + 8, 8 * mx:8 * mx + 8]
    want = port.decode_single_block(blocks[i], qs[2].astype(np.float32))      # Cb with Cr's table (loadjpg.cpp:984)
    assert np.array_equal(cb, want)
    assert not np.array_equal(cb, port.decode_single_block(blocks[i], qs[1].astype(np.float32)))
