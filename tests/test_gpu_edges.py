"""GPU tests: the adversarial IDCT blocks (tests/golden/idct_edges.npz) and worst-case entropy symbols, through every
kernel variant, bit for bit against the oracle.

The blocks sit where the kernels decide per block or per sample: fast results the error window must catch, samples
near an integer, both sides of every precondition of the tensor-core fast tier, the DC-only shortcut, the
short-block switch of the CUDA-core kernel.  They are placed in Y, Cb and Cr of images of every sampling, in warps
whose lanes disagree, in quantities that overflow the per-warp list of exact re-evaluations, and under three
distinct quantisation tables (Cb is de-quantised with Cr's table, like loadjpg.cpp:984)."""
import numpy as np
import pytest

from tests import cases
from tests import jpeg_writer as jw
from tools.gen_jpegs import encode_jpeg, synth_rgb
from tools.make_idct_edges import QUANT

pytestmark = pytest.mark.gpu

FLAG_SETS = ("default", "tensor_core", "cuda_core", "keep_planes", "bmp", "bmp_tensor_core")


def _flags(hjd, name):
    return {"default": 0, "tensor_core": hjd.FLAG_TENSOR_CORE_IDCT, "cuda_core": hjd.FLAG_CUDA_CORE_IDCT,
            "keep_planes": hjd.FLAG_KEEP_PLANES, "bmp": hjd.FLAG_BMP_OUT,
            "bmp_tensor_core": hjd.FLAG_BMP_OUT | hjd.FLAG_TENSOR_CORE_IDCT}[name]


def _expected_variant(name):
    """idct_variant: bit 0 = tensor-core fused kernel ran, bit 1 = CUDA-core fused kernel; 0 = the unfused planes
    kernel.  These images are small, so the default picks the CUDA-core kernel."""
    return {"default": 2, "tensor_core": 1, "cuda_core": 2, "keep_planes": 0, "bmp": 2, "bmp_tensor_core": 1}[name]


def _template(sampling, w, h, seed=1):
    if sampling == "gray":
        return encode_jpeg(synth_rgb(w, h, seed), 50, gray=True)
    if sampling == "440":
        return cases.encode_jpeg_cv(synth_rgb(w, h, seed), 50, "440")
    return encode_jpeg(synth_rgb(w, h, seed), 50, {"444": "4:4:4", "422": "4:2:2", "420": "4:2:0"}[sampling])


def _comp_order(g):
    """[(component, block index, MCU)] of every block in scan order."""
    ncomp = g["ncomp"]
    ny = g["hf"] * g["vf"] if ncomp == 3 else 1
    bpm = ny + 2 if ncomp == 3 else 1
    out = []
    for m in range(g["mcus_x"] * g["mcus_y"]):
        for b in range(bpm):
            out.append((0 if b < ny else b - ny + 1, m * bpm + b, m))
    return out


def _bridge_dc(coef, g, placed, restart_interval):
    """Give the blocks that were not placed a DC that keeps every DC difference within category 11 (the standard
    tables' largest), so that placed blocks with DC up to +-2048 can follow each other."""
    order = _comp_order(g)
    for comp in range(g["ncomp"]):
        seq = [(bi, m) for c, bi, m in order if c == comp]
        prev, prev_m = 0, -1
        for j, (bi, m) in enumerate(seq):
            if restart_interval and m != prev_m and m % restart_interval == 0:
                prev = 0
            if not placed[bi]:
                nxt = 0
                if j + 1 < len(seq):
                    nbi, nm = seq[j + 1]
                    if placed[nbi] and not (restart_interval and nm != m and nm % restart_interval == 0):
                        nxt = int(coef[nbi, 0])
                coef[bi, 0] = int(np.clip(0, max(prev, nxt) - 2047, min(prev, nxt) + 2047))
            prev, prev_m = int(coef[bi, 0]), m


def _place(template, blocks, tq_tables, restart_interval=0, every=3, offset=0):
    """A file of `template`'s size and sampling whose blocks (every `every`-th of each component, first at `offset`)
    are `blocks` in turn; tq_tables: the quantisation table (zig-zag) of each component.  With every >= 3 the two
    blocks in between bridge any pair of DCs in [-2048, 2048]."""
    from oracle import port
    g = port.decode(template, entropy_only=True)["geometry"]
    coef = np.zeros((g["blocks"], 64), dtype=np.int64)
    placed = np.zeros(g["blocks"], dtype=bool)
    k = 0
    seen = {}
    first = {}
    for comp, bi, m in _comp_order(g):
        j = seen.get(comp, 0)
        seen[comp] = j + 1
        after_reset = first.setdefault((comp, m), bi) == bi and (m == 0 or (restart_interval and m % restart_interval == 0))
        if (j + offset) % every == 0:
            if after_reset and abs(int(blocks[k % len(blocks)][0])) > 2047:
                continue                    # a DC difference of 2048 from the reset predictor has no code: next slot
            coef[bi] = blocks[k % len(blocks)]
            placed[bi] = True
            k += 1
    _bridge_dc(coef, g, placed, restart_interval)
    quant, tq = {}, []
    for t in tq_tables:
        key = next((i for i, q in quant.items() if np.array_equal(q, t)), len(quant))
        quant[key] = t
        tq.append(key)
    return jw.blocks_to_jpeg(template, coef, g, quant, tq=tq[:g["ncomp"]], restart_interval=restart_interval)


def _edges():
    import os
    d = np.load(os.path.join(os.path.dirname(__file__), "golden", "idct_edges.npz"))
    return d["coef"].astype(np.int64), d["qidx"].astype(np.int64), d["label"]


def idct_images():
    coef, qidx, label = _edges()
    files = {}
    # placement: every table's blocks in Y, Cb and Cr of every sampling; MCU counts that are not multiples of 128
    sizes = {"444": (72, 56), "422": (136, 40), "420": (136, 72), "440": (72, 112), "gray": (200, 64)}
    for t in range(len(QUANT)):
        blk = coef[qidx == t]
        for s, (w, h) in sizes.items():
            for off in (0, 1, 2):
                files[f"place_q{t}_{s}_{off}"] = _place(_template(s, w, h, seed=t + 3), blk, [QUANT[t]] * 3,
                                                        restart_interval=(0, 3, 1)[off], offset=off)
    # lane control: a warp of 32 gray blocks (one lane each) that end at <= 20 with one lane at 21, and the reverse
    b20, b21 = coef[(label == "last_20") & (qidx == 0)], coef[(label == "last_21") & (qidx == 0)]
    lanes = []
    for warp in range(4):
        for lane in range(32):
            odd = lane == (5 + 9 * warp) % 32
            short = (warp % 2 == 0) != odd
            lanes.append((b20 if short else b21)[(warp + lane) % len(b20)])
    files["lanes_gray"] = _place(_template("gray", 8 * 128, 8), np.array(lanes), [QUANT[0]], every=1)
    files["lanes_444"] = _place(_template("444", 8 * 128, 8), np.array(lanes), [QUANT[0]] * 3, every=1)
    # exact-list pressure: every lane with a row of 8 flagged samples; all-exact lanes among fast-tier lanes, and a
    # last unit of 128 MCUs that is partly beyond the image
    rows = coef[label == "row_flagged"]
    files["pressure_rows"] = _place(_template("gray", 8 * 64, 16), rows, [QUANT[0]], every=1)
    mix = []
    for i in range(200):
        lab = ("ac_range_out", "tc_fast_wrong", "row_flagged", "a_above", "cc_fast_wrong")[i % 5]
        pool = coef[(label == lab) & (qidx == 0)]
        mix.append(pool[i % len(pool)])
    files["pressure_mixed"] = _place(_template("gray", 8 * 200, 8), np.array(mix), [QUANT[0]], every=1)
    files["pressure_mixed_420"] = _place(_template("420", 16 * 67, 16), np.array(mix), [QUANT[0]] * 3, every=1)
    # three distinct tables: Cb is de-quantised with Cr's
    three = [QUANT[3], QUANT[1], np.clip(QUANT[3] // 3 + 1, 1, 255).astype(np.uint8)]
    blk = coef[np.isin(label, ["last_20", "last_21", "near_sat_127", "dc_plus_1", "near_integer"])]
    for s, (w, h) in (("420", (64, 48)), ("444", (40, 24)), ("422", (48, 32))):
        for ri in (0, 2):
            files[f"three_tables_{s}_ri{ri}"] = _place(_template(s, w, h), blk, three, restart_interval=ri, every=1)
    return files


def tiny_images():
    """Many tiny images of mixed sampling in one batch: units of 128 MCUs span images (the kernels' look-up mode)."""
    coef, qidx, label = _edges()
    blk = coef[qidx == 0]
    out = []
    for i in range(48):
        s = ("444", "420", "gray", "422", "440")[i % 5]
        w, h = 8 + 8 * (i % 3), 8 + 8 * ((i // 3) % 2)
        out.append(_place(_template(s, w, h, seed=100 + i), np.roll(blk, -7 * i, axis=0), [QUANT[0]] * 3, every=2,
                          offset=i % 2))
    return out


# ---- entropy worst case ---------------------------------------------------------------------------------------
AC_SYMBOLS = [0x00, 0xF0] + [(r << 4) | s for r in range(16) for s in range(1, 11)]


def _long_tables(dc16=False):
    """AC: every size-10 symbol a 16-bit code, the rest 8 bits.  DC: categories 0-10 4 bits, 11 a 15-bit code
    (16 bits with dc16: loadjpg.cpp:562 searches up to 15)."""
    short = [s for s in AC_SYMBOLS if (s & 15) != 10]
    long_ = [s for s in AC_SYMBOLS if (s & 15) == 10]
    ac_bits = [0] * 16
    ac_bits[7], ac_bits[15] = len(short), len(long_)
    dc_bits = [0] * 16
    dc_bits[3] = 11
    dc_bits[15 if dc16 else 14] = 1
    ac, dc = (ac_bits, short + long_), (dc_bits, list(range(12)))
    return {(0, 0): dc, (0, 1): dc, (1, 0): ac, (1, 1): ac}


def _worst_blocks(n, rng):
    """63 AC coefficients of magnitude 512-1023 (26 bits each with the tables above), DCs whose differences are
    category 11, ZRL chains that end at index 63, blocks whose last coefficient is at 63 (no EOB)."""
    out = np.zeros((n, 64), dtype=np.int64)
    for i in range(n):
        kind = i % 4
        if kind in (0, 1):
            out[i, 1:] = rng.integers(512, 1024, size=63) * rng.choice([-1, 1], size=63)
        elif kind == 2:
            out[i, 63] = int(rng.integers(512, 1024))            # 62 zeros: three ZRLs, then run 14
            out[i, 1] = int(rng.integers(-1023, -511))
        else:
            pos = [1, 18, 35, 52, 63]                           # runs of 16: ZRL then a run-0 symbol
            out[i, pos] = rng.integers(512, 1024, size=len(pos))
    return out


def entropy_images(dc16=False):
    from oracle import port
    rng = np.random.default_rng(11)
    files = {}
    for s, (w, h) in (("420", (64, 64)), ("444", (32, 40)), ("gray", (48, 48))):
        t = _template(s, w, h)
        g = port.decode(t, entropy_only=True)["geometry"]
        coef = _worst_blocks(g["blocks"], rng)
        k = {}
        for comp, bi, m in _comp_order(g):               # DC differences of category 11: 0, 1500, 0, -1500, ... per component
            j = k.get(comp, 0)
            k[comp] = j + 1
            coef[bi, 0] = (0, 1500, 0, -1500)[j % 4]
        for ri in ((0,) if dc16 else (0, 1, 3, 8)):
            files[f"entropy_{s}_ri{ri}"] = jw.blocks_to_jpeg(t, coef, g, {0: QUANT[0]}, tq=[0, 0, 0][:g["ncomp"]],
                                                             tables=_long_tables(dc16), restart_interval=ri)
    return files


def _decode_all(hjd, files, flags):
    with hjd.BatchDecoder(0, flags) as d:
        d.upload(files)
        d.decode()
        st = d.status().copy()
        out = dict(status=st, variant=d.idct_variant, rounds=d.selfsync_rounds, coef=[], rgb=[], planes=[], bmp=[])
        coef = d.coefficients()
        slab = d.plane_slab() if flags & hjd.FLAG_KEEP_PLANES else None
        for i in range(len(files)):
            out["coef"].append(d.image_coefficients(i, coef).copy())
            if flags & hjd.FLAG_BMP_OUT:
                out["bmp"].append(d.bmp(i))
            else:
                out["rgb"].append(d.rgb(i).copy())
            if slab is not None:
                out["planes"].append([None if p is None else p.copy() for p in d.planes(i, slab)])
    return out


def _check(port, names, files, want, got, name):
    assert (got["status"] == 0).all(), (name, got["status"])
    assert got["variant"] == _expected_variant(name), (name, got["variant"])
    for i, n in enumerate(names):
        w = want[n]
        assert np.array_equal(got["coef"][i], w["coef"]), (name, n, "coefficients")
        if got["bmp"]:
            assert got["bmp"][i] == port.bmp24_bytes(w["rgb"]), (name, n, "bmp")
        else:
            assert np.array_equal(got["rgb"][i], w["rgb"]), (name, n, "rgb")
        if got["planes"]:
            for a, b in zip(got["planes"][i], w["planes"]):
                if a is not None:
                    assert np.array_equal(a, b), (name, n, "planes")


@pytest.fixture(scope="module")
def decoded(hjd, port):
    """Every image of the module under every flag set, with the oracle's answers."""
    batches = {"idct": idct_images(), "tiny": {f"tiny_{i}": f for i, f in enumerate(tiny_images())},
               "entropy": entropy_images()}
    want = {}
    for files in batches.values():
        for n, f in files.items():
            want[n] = port.decode(f)
            assert want[n]["rc"] == 0, n
    from oracle import refbind
    if refbind.available("std"):                                 # the oracle is the reference here too
        for files in batches.values():
            for n, f in files.items():
                r = refbind.decode(f, mode=1)
                assert r["rc"] == 0 and np.array_equal(r["coef"], want[n]["coef"]), n
                assert np.array_equal(r["rgb"], want[n]["rgb"]), n
    got = {}
    for b, files in batches.items():
        for name in FLAG_SETS:
            got[(b, name)] = _decode_all(hjd, list(files.values()), _flags(hjd, name))
    return batches, want, got


@pytest.mark.parametrize("flag_set", FLAG_SETS)
@pytest.mark.parametrize("batch", ["idct", "tiny", "entropy"])
def test_edge_blocks_bit_exact(decoded, port, batch, flag_set):
    batches, want, got = decoded
    names = list(batches[batch])
    _check(port, names, batches[batch], want, got[(batch, flag_set)], flag_set)


def test_entropy_worst_case_paths(hjd, port, decoded):
    """Blocks longer than a 1024-bit sub-sequence: the restart-free files go through the self-synchronising kernel
    (it needs more than the confirming round), and the single-thread path gives the same answers."""
    batches, want, got = decoded
    files = batches["entropy"]
    assert got[("entropy", "default")]["rounds"] >= 2
    for n, f in files.items():
        if n.endswith("_ri0"):
            assert hjd.probe(f)[1].scan_bytes >= 1024, n
    nss = _decode_all(hjd, list(files.values()), hjd.FLAG_NO_SELFSYNC)
    _check(port, list(files), files, want, nss, "default")


def test_sixteen_bit_dc_code_on_worst_case_blocks(hjd, port):
    """The same worst-case blocks with DC category 11 at a 16-bit code (beyond loadjpg.cpp:562): the oracle with its
    16-bit switch is the checker."""
    files = entropy_images(dc16=True)
    try:
        port.set_dc16(True)
        want = {n: port.decode(f) for n, f in files.items()}
    finally:
        port.set_dc16(False)
    for flags in (0, hjd.FLAG_NO_SELFSYNC, hjd.FLAG_TENSOR_CORE_IDCT):
        got = _decode_all(hjd, list(files.values()), flags)
        assert (got["status"] == 0).all(), got["status"]
        for i, n in enumerate(files):
            assert np.array_equal(got["coef"][i], want[n]["coef"]), (flags, n)
            assert np.array_equal(got["rgb"][i], want[n]["rgb"]), (flags, n)
