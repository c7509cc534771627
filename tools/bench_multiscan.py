"""Timing of the multi-scan path (HJD_FLAG_MULTI_SCAN) on one GPU; one JSON line per workload and round.

    W1  1024 x 1920x1080 4:2:0 q85, progressive with libjpeg's default script, no restart markers
    W2  the same with restart markers (restart_marker_blocks=8)
    W3  their baseline twins (same pixels, same coefficients)
    W4  single-image latency of one W1 file

Per workload: ms per step (CUDA events via BatchDecoder.mark / elapsed_ms over K steps after a warm-up; the
workloads alternate round by round), MP/s, the entropy / IDCT+colour split of one serial decode, launches, and the
host upload time (parse incl. the walk over every scan + metadata + H2D, host clock around a synchronised upload).
The device name and power limit are read in the same run.

    python tools/bench_multiscan.py --images 1024 --steps 10 --warmup 3 --rounds 3 --out profiles/x.jsonl
"""
from __future__ import annotations

import argparse
import io
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from PIL import Image  # noqa: E402

from tools.gen_jpegs import synth_rgb_fast  # noqa: E402


def _encode(args):
    i, progressive, restart = args
    buf = io.BytesIO()
    kw = dict(format="JPEG", quality=85, subsampling=2, progressive=progressive)
    if restart:
        kw["restart_marker_blocks"] = restart
    Image.fromarray(synth_rgb_fast(1920, 1080, i)).save(buf, **kw)
    return buf.getvalue()


def make(n, progressive, restart):
    with ProcessPoolExecutor(max_workers=min(os.cpu_count() or 1, 32)) as ex:
        return list(ex.map(_encode, [(i, progressive, restart) for i in range(n)], chunksize=8))


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import hls_jpeg_decoder_b200 as hjd

    if hjd.lib().hjd_device_count() < 1:
        raise SystemExit("no CUDA device: nothing measured")
    dev = device_line()
    work = {"W1": make(a.images, True, 0), "W2": make(a.images, True, 8), "W3": make(a.images, False, 0)}
    work["W4"] = work["W1"][:1]
    decs, info = {}, {}
    for name, files in work.items():
        dec = hjd.BatchDecoder(0, hjd.FLAG_MULTI_SCAN)
        dec.set_overlap(0)                                   # one stream: per-stage timings
        ups = []
        for _ in range(3):
            t0 = time.perf_counter()
            dec.upload(files)                                # parses, copies and synchronises
            ups.append((time.perf_counter() - t0) * 1e3)
        for _ in range(a.warmup):
            dec.decode()
        dec.sync()
        st = dec.status()
        assert (st == 0).all(), (name, st[st != 0][:8])
        dec.decode()
        t = dec.timings()
        info[name] = dict(upload_ms=min(ups), entropy_ms=t["scan_ms"] + t["entropy_ms"],
                          idct_color_ms=t["idct_ms"] + t["color_ms"], launches=t["launches"],
                          pixels=dec.pixels, scan_bytes=dec.scan_bytes,
                          scans=sum(dec.num_scans(i) for i in range(len(files))))
        decs[name] = dec
    lines = []
    for r in range(a.rounds):
        for name, dec in decs.items():
            for _ in range(a.warmup):
                dec.decode()
            dec.mark(0)
            for _ in range(a.steps):
                dec.decode()
            dec.mark(1)
            ms = dec.elapsed_ms(0, 1) / a.steps
            line = dict(workload=name, round=r, images=len(work[name]), ms_per_step=round(ms, 4),
                        mp_per_s=round(info[name]["pixels"] / 1e6 / (ms / 1e3), 1), device=dev,
                        **{k: (round(v, 4) if isinstance(v, float) else v) for k, v in info[name].items()})
            print(json.dumps(line), flush=True)
            lines.append(line)
    if a.out:
        with open(a.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")
    for dec in decs.values():
        dec.close()


if __name__ == "__main__":
    main()
