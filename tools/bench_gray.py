"""Timing of the luma-only decode (FLAG_GRAY_OUT) on one GPU; one JSON line per measurement.

    G1  HBM-resident, 1024 x 1920x1080 4:2:0 q85 Ri=8 (config 2, tools/gen_jpegs.py): ms per step (CUDA events over K
        steps, the variants alternating round by round) of RGB (default: the tensor-core fused kernel on this batch),
        RGB through the CUDA-core fused kernel, gray, and gray at 1/2, 1/4 and 1/8; and the entropy / IDCT split of one
        serial decode, whose IDCT stage is the luma kernel's time (gray) or the fused RGB kernel's (RGB)
    G2  the same files end to end through pinned host buffers (decode_host), RGB and gray: source MP/s and output GB/s,
        beside the ceiling hjd_link_probe measures for the same H2D and D2H bytes
    G3  bench_multiscan's W2 (progressive 1080p with restart markers) in RGB and in gray, and the scans read
    G4  bench.py (config 2) of this tree and of --parent DIR (a built checkout of another commit), alternated

The device name and power limit are read in the same run.

    python tools/bench_gray.py --steps 10 --warmup 3 --rounds 3 --parent ../parent --out profiles/x.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools import gen_jpegs  # noqa: E402
from tools.bench_multiscan import device_line, make  # noqa: E402

LINES = []


def emit(**kw):
    line = {k: (round(v, 4) if isinstance(v, float) else v) for k, v in kw.items()}
    print(json.dumps(line), flush=True)
    LINES.append(line)


def variants(hjd):
    g = hjd.FLAG_GRAY_OUT
    return {"rgb": 0, "rgb_cuda_core": hjd.FLAG_CUDA_CORE_IDCT, "gray": g, "gray_1/2": g | hjd.FLAG_SCALE_1_2,
            "gray_1/4": g | hjd.FLAG_SCALE_1_4, "gray_1/8": g | hjd.FLAG_SCALE_1_8}


def g1(hjd, files, a, dev):
    decs, split = {}, {}
    for name, flags in variants(hjd).items():
        dec = hjd.BatchDecoder(0, flags)
        dec.set_overlap(0)                                   # one stream: per-stage timings
        dec.upload(files)
        for _ in range(a.warmup):
            dec.decode()
        st = dec.status()
        assert (st == 0).all(), st[st != 0][:8]
        dec.decode()
        t = dec.timings()
        split[name] = dict(entropy_ms=t["scan_ms"] + t["entropy_ms"], idct_ms=t["idct_ms"], color_ms=t["color_ms"],
                           idct_variant=dec.idct_variant, out_bytes=dec.rgb_bytes)
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
            emit(bench="G1", variant=name, round=r, images=len(files), ms_per_step=ms,
                 source_mp_per_s=dec.pixels / 1e6 / (ms / 1e3), device=dev, **split[name])
    # the IDCT stage alone, many serial decodes per variant, alternating: the kernel's time on this batch
    stage = {name: [] for name in decs}
    for r in range(a.rounds * 3):
        for name, dec in decs.items():
            dec.decode()
            stage[name].append(dec.timings()["idct_ms"])
    for name, v in stage.items():
        v.sort()
        emit(bench="G1 stage", variant=name, images=len(files), idct_ms_median=v[len(v) // 2], idct_ms_min=v[0],
             samples=len(v), idct_variant=split[name]["idct_variant"], device=dev)
    for dec in decs.values():
        dec.close()


def g2(hjd, files, a, dev):
    arena = hjd.PinnedArena(files, device=0)
    pixels = None
    for name in ("rgb", "gray"):
        flags = variants(hjd)[name]
        cap = int(hjd.lib().hjd_out_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n, flags))
        out = hjd.lib().hjd_host_alloc_near(0, cap)
        with hjd.BatchDecoder(0, flags) as dec:
            dec.decode_host(arena, out, cap)                 # warm-up (allocations, module loads)
            pixels = dec.pixels
            times = []
            for _ in range(a.e2e_steps):
                t0 = time.perf_counter()
                _, st = dec.decode_host(arena, out, cap)
                times.append(time.perf_counter() - t0)
            assert (st == 0).all()
        ms_h2d, ms_d2h = hjd.link_probe(0, arena.ptr, arena.bytes, out, cap, reps=3)
        t = min(times)
        t_link = max(ms_h2d, ms_d2h) / 1e3
        emit(bench="G2", variant=name, images=len(files), ms_per_call=t * 1e3, source_mp_per_s=pixels / 1e6 / t,
             out_gb_per_s=cap / 1e9 / t, h2d_bytes=arena.bytes, d2h_bytes=cap,
             link_ceiling_ms=t_link * 1e3, link_ceiling_mp_per_s=pixels / 1e6 / t_link,
             frac_of_link_ceiling=t_link / t, device=dev)
        hjd.lib().hjd_host_free(out)
    arena.close()


def g3(hjd, a, dev):
    files = make(a.images, True, 8)
    for name, flags in (("W2 rgb", hjd.FLAG_MULTI_SCAN), ("W2 gray", hjd.FLAG_MULTI_SCAN | hjd.FLAG_GRAY_OUT)):
        with hjd.BatchDecoder(0, flags) as dec:
            dec.set_overlap(0)
            dec.upload(files)
            dec.decode()
            assert (dec.status() == 0).all()
            dec.decode()
            t = dec.timings()
            dec.mark(0)
            for _ in range(a.steps):
                dec.decode()
            dec.mark(1)
            ms = dec.elapsed_ms(0, 1) / a.steps
            emit(bench="G3", workload=name, images=len(files), steps=a.steps, ms_per_step=ms,
                 source_mp_per_s=dec.pixels / 1e6 / (ms / 1e3), entropy_ms=t["scan_ms"] + t["entropy_ms"],
                 idct_ms=t["idct_ms"], color_ms=t["color_ms"], launches=t["launches"],
                 scans=sum(dec.num_scans(i) for i in range(len(files))),
                 scans_in_files=sum(len(hjd.scans(f)) for f in files), device=dev)


def g4(a, dev):
    trees = {"this": ROOT, "parent": os.path.abspath(a.parent)}
    for r in range(a.rounds):
        for name, tree in trees.items():
            p = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(a.steps), "--warmup",
                                str(a.warmup), "--no-cpu-baseline", "--no-extras"], cwd=tree, capture_output=True,
                               text=True)
            rec = next((json.loads(x) for x in p.stdout.splitlines() if x.startswith("{")), None)
            if rec is None:
                raise SystemExit(f"bench.py in {tree} failed:\n{p.stdout[-2000:]}\n{p.stderr[-2000:]}")
            emit(bench="G4", tree=name, round=r, value=rec["value"], unit=rec["unit"], ms_per_step=rec["ms_per_step"],
                 device=dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--parent", default=None, help="built checkout of the commit to compare bench.py with (G4)")
    ap.add_argument("--only", default="G1,G2,G3,G4")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import hls_jpeg_decoder_b200 as hjd

    if hjd.lib().hjd_device_count() < 1:
        raise SystemExit("no CUDA device: nothing measured")
    dev = device_line()
    only = set(a.only.split(","))
    files = gen_jpegs.make_batch("c2", a.images) if only & {"G1", "G2"} else None
    if "G1" in only:
        g1(hjd, files, a, dev)
    if "G2" in only:
        g2(hjd, files, a, dev)
    if "G3" in only:
        g3(hjd, a, dev)
    if "G4" in only and a.parent:
        g4(a, dev)
    if a.out:
        with open(a.out, "w") as fh:
            for line in LINES:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
