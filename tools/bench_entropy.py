"""The restart-interval entropy kernel (kernel 1a) of two or more library builds, alternated; one JSON line per measurement.

Every build decodes every workload in its own process (HJD_LIB_PATH selects the build), round by round, the builds
alternating within a round.  Per (build, workload, round):
    entropy_ms   median of the entropy stage (marker scan excluded) over --serial serial decodes on one stream
    scan_ms      median of the marker scan over the same decodes
    ms_per_step  CUDA events over --steps HBM-resident steps after --warmup steps (the decode bench.py times)
    coef_xor / coef_sum   a fold of the whole coefficient slab: every build must give the same one
Workloads (bench.py's): c2, c2q50, c2q95, c5 (8192 thumbnails), and shard128 (the 128-image rank-0 shard of one c2
batch cut over 8 GPUs, bench.py's "strong" sub-record).  The card's name, power limit and SM clocks are read in
the same run.

    python tools/bench_entropy.py --lib parent=/path/to/parent/libhjd.so --lib this= --rounds 3 --out profiles/x.jsonl

(an empty path is this tree's hls_jpeg_decoder_b200/libhjd.so).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {"c2": ("c2", 1024, 1, "weak"), "c2q50": ("c2q50", 1024, 1, "weak"), "c2q95": ("c2q95", 1024, 1, "weak"),
             "c5": ("c5", 8192, 1, "weak"), "shard128": ("c2", 1024, 8, "strong")}


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def worker(a):
    import numpy as np
    import bench
    import hls_jpeg_decoder_b200 as hjd

    if hjd.lib().hjd_device_count() < 1:
        raise SystemExit("no CUDA device: nothing measured")
    config, n, world, scaling = WORKLOADS[a.worker]
    files = bench.load_images(n, 0, world, config, scaling)
    arena = hjd.PinnedArena(files)
    rec = {"workload": a.worker, "images": len(files)}
    with hjd.BatchDecoder(0) as dec:
        dec.set_overlap(0)                                   # one stream: per-stage timings
        dec.upload_arena(arena)
        for _ in range(a.warmup):
            dec.decode()
        st = dec.status()
        assert (st == 0).all(), st[st != 0][:8]
        ent, scan = [], []
        for _ in range(a.serial):
            dec.decode()
            t = dec.timings()
            ent.append(t["entropy_ms"])
            scan.append(t["scan_ms"])
        rec.update(entropy_ms=float(np.median(ent)), entropy_ms_min=min(ent), scan_ms=float(np.median(scan)))
        v = dec.coefficients().view(np.uint64)
        rec.update(coef_xor=hex(int(np.bitwise_xor.reduce(v, axis=None))), coef_sum=hex(int(v.sum(dtype=np.uint64))))
    with hjd.BatchDecoder(0) as dec:                         # bench.py's decoder: default settings
        dec.upload_arena(arena)
        dec.sync()
        for _ in range(a.warmup):
            dec.decode()
        dec.mark(0)
        for _ in range(a.steps):
            dec.decode()
        dec.mark(1)
        dec.sync()
        rec["ms_per_step"] = dec.elapsed_ms(0, 1) / a.steps
    arena.close()
    print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="NAME=PATH of a libhjd.so build (empty PATH: this tree's)")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--serial", type=int, default=15)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    libs = [x.split("=", 1) for x in a.lib] or [["this", ""]]
    lines = []

    def emit(**kw):
        line = {k: (round(v, 4) if isinstance(v, float) else v) for k, v in kw.items()}
        print(json.dumps(line), flush=True)
        lines.append(line)

    emit(device=device_line(), libs={name: path or "tree" for name, path in libs})
    coef = {}
    for r in range(a.rounds):
        for wl in a.workloads.split(","):
            for name, path in libs:
                env = dict(os.environ)
                env.pop("HJD_LIB_PATH", None)
                if path:
                    env["HJD_LIB_PATH"] = os.path.abspath(path)
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", wl, "--steps", str(a.steps),
                                    "--warmup", str(a.warmup), "--serial", str(a.serial)], cwd=ROOT, env=env,
                                   capture_output=True, text=True)
                rec = next((json.loads(x) for x in p.stdout.splitlines() if x.startswith("{")), None)
                if rec is None:
                    raise SystemExit(f"{name} on {wl} failed:\n{p.stdout[-2000:]}\n{p.stderr[-2000:]}")
                fold = (rec.pop("coef_xor"), rec.pop("coef_sum"))
                same = coef.setdefault(wl, fold) == fold
                emit(build=name, round=r, **rec, coef_same_as_first=same, device=device_line())
                if not same:
                    raise SystemExit(f"{name} on {wl}: coefficient slab differs from the first build's")
    if a.out:
        with open(a.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
