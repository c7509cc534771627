"""Timing of the EXIF orientation pass (FLAG_EXIF_ORIENT) on one GPU; one JSON line per measurement.

Input: config 2 (1024 x 1920x1080 4:2:0 q85 Ri=8, tools/gen_jpegs.py) with an Exif APP1 spliced after every SOI that
states orientation 6 (rotate 90 degrees clockwise, what a phone writes for a portrait photo), against the same files
with an APP1 that states 1 (same file sizes; no staging, no pass).  Every batch is created with FLAG_EXIF_ORIENT.

    O1  HBM-resident ms per step (CUDA events over K steps, the variants alternating round by round): RGB and gray, each
        with o = 1 and o = 6; and the IDCT (output) stage of many serial decodes, which holds the orientation pass
    O2  the orientation pass's own time: the median IDCT stage of o = 6 minus that of o = 1, and its bytes (one read
        and one write of the oriented output) over that time, beside a device-to-device cudaMemcpyAsync of the same
        byte count (torch's copy_ of a contiguous uint8 tensor) timed with CUDA events in the same run
    O3  the same files end to end through pinned host buffers (decode_host), RGB with o = 1 and o = 6: source MP/s
    O4  bench.py (config 2) of this tree and of --parent DIR (a built checkout of another commit), alternated

The device name and power limit are read in the same run.

    python tools/bench_orient.py --steps 10 --warmup 3 --rounds 3 --parent ../parent --out profiles/x.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import exif_writer as ew  # noqa: E402
from tools import gen_jpegs  # noqa: E402
from tools.bench_gray import LINES, emit, g4  # noqa: E402
from tools.bench_multiscan import device_line  # noqa: E402


def variants(hjd):
    o = hjd.FLAG_EXIF_ORIENT
    return {"rgb o=1": (o, 1), "rgb o=6": (o, 6), "gray o=1": (o | hjd.FLAG_GRAY_OUT, 1), "gray o=6": (o | hjd.FLAG_GRAY_OUT, 6)}


def o1_o2(hjd, tagged, a, dev):
    decs = {}
    for name, (flags, o) in variants(hjd).items():
        dec = hjd.BatchDecoder(0, flags)
        dec.set_overlap(0)                                   # one stream: per-stage timings
        dec.upload(tagged[o])
        dec.decode()
        st = dec.status()
        assert (st == 0).all(), st[st != 0][:8]
        assert dec.orientation(0) == o and dec.out_size(0) == ((1080, 1920) if o == 6 else (1920, 1080))
        decs[name] = dec
    for r in range(a.rounds):
        for name, dec in decs.items():
            for _ in range(a.warmup):
                dec.decode()
            dec.mark(0)
            for _ in range(a.steps):
                dec.decode()
            dec.mark(1)
            ms = dec.elapsed_ms(0, 1) / a.steps
            emit(bench="O1", variant=name, round=r, images=len(tagged[1]), ms_per_step=ms,
                 source_mp_per_s=dec.pixels / 1e6 / (ms / 1e3), launches=dec.timings()["launches"], device=dev)
    stage = {name: [] for name in decs}
    for r in range(a.rounds * 5):
        for name, dec in decs.items():
            dec.decode()
            stage[name].append(dec.timings()["idct_ms"])
    med = {}
    for name, v in stage.items():
        v.sort()
        med[name] = v[len(v) // 2]
        emit(bench="O1 stage", variant=name, images=len(tagged[1]), idct_ms_median=med[name], idct_ms_min=v[0],
             samples=len(v), idct_variant=decs[name].idct_variant, device=dev)
    import torch
    for kind in ("rgb", "gray"):
        nbytes = decs[f"{kind} o=6"].rgb_bytes
        src = torch.empty(nbytes, dtype=torch.uint8, device="cuda:0")
        dst = torch.empty_like(src)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(3):
            dst.copy_(src)
        ts = []
        for _ in range(a.rounds * 5):
            ev[0].record()
            dst.copy_(src)
            ev[1].record()
            ev[1].synchronize()
            ts.append(ev[0].elapsed_time(ev[1]))
        ts.sort()
        copy_ms = ts[len(ts) // 2]
        pass_ms = med[f"{kind} o=6"] - med[f"{kind} o=1"]
        emit(bench="O2", variant=kind, images=len(tagged[1]), oriented_bytes=nbytes, pass_ms=pass_ms,
             pass_gb_per_s=2 * nbytes / 1e9 / (pass_ms / 1e3), pass_us_per_image=pass_ms * 1e3 / len(tagged[1]),
             d2d_copy_ms=copy_ms, d2d_copy_gb_per_s=2 * nbytes / 1e9 / (copy_ms / 1e3), pass_over_copy=pass_ms / copy_ms,
             note="bytes: one read + one write of the oriented output; pass = median IDCT stage o=6 minus o=1", device=dev)
        del src, dst
    for dec in decs.values():
        dec.close()


def o3(hjd, tagged, a, dev):
    for o in (1, 6):
        flags = hjd.FLAG_EXIF_ORIENT
        arena = hjd.PinnedArena(tagged[o], device=0)
        cap = int(hjd.lib().hjd_out_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n, flags))
        out = hjd.lib().hjd_host_alloc_near(0, cap)
        with hjd.BatchDecoder(0, flags) as dec:
            dec.decode_host(arena, out, cap)                 # warm-up (allocations, module loads)
            times = []
            for _ in range(a.e2e_steps):
                t0 = time.perf_counter()
                _, st = dec.decode_host(arena, out, cap)
                times.append(time.perf_counter() - t0)
            assert (st == 0).all()
            t = min(times)
            emit(bench="O3", variant=f"rgb o={o}", images=arena.n, ms_per_call=t * 1e3,
                 source_mp_per_s=dec.pixels / 1e6 / t, out_gb_per_s=cap / 1e9 / t, device=dev)
        hjd.lib().hjd_host_free(out)
        arena.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--parent", default=None, help="built checkout of the commit to compare bench.py with (O4)")
    ap.add_argument("--only", default="O1,O3,O4")
    ap.add_argument("--out", default=None, help="JSON lines appended here")
    a = ap.parse_args()
    import hls_jpeg_decoder_b200 as hjd

    if hjd.lib().hjd_device_count() < 1:
        raise SystemExit("no CUDA device: nothing measured")
    dev = device_line()
    only = set(a.only.split(","))
    if only & {"O1", "O3"}:
        files = gen_jpegs.make_batch("c2", a.images)
        tagged = {o: [ew.with_orientation(f, o) for f in files] for o in (1, 6)}
        if "O1" in only:
            o1_o2(hjd, tagged, a, dev)
        if "O3" in only:
            o3(hjd, tagged, a, dev)
    if "O4" in only and a.parent:
        g4(a, dev)
        for line in LINES:                                   # bench_gray's comparison, under this tool's name
            if line["bench"] == "G4":
                line["bench"] = "O4"
    if a.out:
        with open(a.out, "a") as fh:
            for line in LINES:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
