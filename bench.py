#!/usr/bin/env python
"""bench.py -- decoded MP/s on a batch of synthetic 1080p 4:2:0 baseline JPEGs (BASELINE.json config 2/3).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle/_ref)

A step = one pass of the whole hot path (marker scan -> entropy decode -> dequant/IDCT -> colour)
over this rank's batch (default 1024 images of 1920x1080 4:2:0 q85 Ri=8, compressed files already
resident in HBM).  Weak scaling: every rank decodes its own 1024-image shard, no collective in the
data path; torch.distributed (NCCL) is used only for the barrier and the max-over-ranks timing.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H = 1920, 1080     # config 2 geometry (the CPU arm always decodes config-2 images)
FALLBACK_HBM_GBS = 6650.0          # /opt/skills/guides/B200_PROFILING.md fallback
DUMP_PIXELS = 4 << 20              # --dump-outputs: sampled RGB pixels over all images (48 MiB as float32)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--images", type=int, default=0, help="images per GPU (default: 1024 for c2, 1 for c4, 8192 for c5)")
    ap.add_argument("--config", default="c2", choices=["c2", "c2nr", "c2q50", "c2q95", "c4", "c5"],
                    help="BASELINE.json workload: c2 = 1080p 4:2:0 Ri=8 batch (headline), c4 = one 8192x8192 4:4:4 "
                         "restart-free image, c5 = 256x256 gray/4:2:0 thumbnails")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank decodes its own batch; strong: one batch sharded over the ranks (config 3)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the sub-records that follow the timed headline (strong scaling of one batch = configs[2], "
                         "configs[3] and configs[4], the oracle-checked parity block)")
    ap.add_argument("--extra-steps", type=int, default=5)
    ap.add_argument("--parity-images", type=int, default=8, help="images per rank checked against the oracle after the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what rank 0's last timed step returned as DIR/<name>.npy: status.npy "
                         "(per image), image_hw.npy (height, width per image) and rgb.npy, float32 [images, S, 3] RGB at S "
                         "pixels per image drawn with a fixed seed (S = %d // images, under 64 MB in all)" % DUMP_PIXELS)
    return ap.parse_args()


def rank_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------
# workload
# ---------------------------------------------------------------------------------------------
WORKLOADS = {
    "c2": dict(n=1024, w=1920, h=1080, desc="synthetic 1920x1080 4:2:0 baseline JPEGs, q85, restart interval 8 MCUs (BASELINE.json configs[1])"),
    "c2nr": dict(n=1024, w=1920, h=1080, desc="synthetic 1920x1080 4:2:0 baseline JPEGs, q85, NO restart markers (restart-free twins of configs[1]): self-synchronising path"),
    "c2q50": dict(n=1024, w=1920, h=1080, desc="synthetic 1920x1080 4:2:0 baseline JPEGs, q50, restart interval 8 MCUs (quality sensitivity of configs[1])"),
    "c2q95": dict(n=1024, w=1920, h=1080, desc="synthetic 1920x1080 4:2:0 baseline JPEGs, q95, restart interval 8 MCUs (quality sensitivity of configs[1])"),
    "c4": dict(n=1, w=8192, h=8192, desc="one synthetic 8192x8192 4:4:4 baseline JPEG, q85, no restart markers: self-synchronising path (BASELINE.json configs[3])"),
    "c5": dict(n=8192, w=256, h=256, desc="synthetic 256x256 thumbnails, even = grayscale, odd = 4:2:0, q75, restart interval 8 MCUs (BASELINE.json configs[4], per-GPU share)"),
}


def load_images(n: int, rank: int, world: int, config: str = "c2", scaling: str = "weak", with_ids: bool = False):
    """Seeded images of one BASELINE.json workload (tools/gen_jpegs), cached on local disk so that
    the ranks of one run (and the reference arm) generate them only once; per user, since other accounts may share
    the temporary directory."""
    import tempfile
    from tools import gen_jpegs
    wl = WORKLOADS[config]
    cache = os.path.join(tempfile.gettempdir(), f"hjd_bench_{os.getuid()}_{config}_{wl['w']}x{wl['h']}_{n}.bin")
    idx = cache + ".idx"
    if not os.path.exists(idx):
        if rank == 0:
            files = [gen_jpegs.make_c4(wl["w"], 4 + i) for i in range(n)] if config == "c4" else gen_jpegs.make_batch(config, n)
            tmp = cache + f".tmp{os.getpid()}"
            with open(tmp, "wb") as fh:
                for f in files:
                    fh.write(f)
            os.replace(tmp, cache)
            with open(idx + ".tmp", "w") as fh:
                json.dump([len(f) for f in files], fh)
            os.replace(idx + ".tmp", idx)
        else:
            t0 = time.time()
            while not os.path.exists(idx):
                time.sleep(0.5)
                if time.time() - t0 > 1800:
                    raise RuntimeError("timed out waiting for rank 0 to generate the images")
    sizes = json.load(open(idx))
    blob = open(cache, "rb").read()
    files, o = [], 0
    for s in sizes:
        files.append(blob[o:o + s])
        o += s
    if scaling == "strong":
        # config 3: ONE batch cut into contiguous image ranges balanced by compressed bytes
        from hls_jpeg_decoder_b200.sharding import shard_range
        lo, hi = shard_range(sizes, rank, world)
        return (files[lo:hi], list(range(lo, hi))) if with_ids else files[lo:hi]
    # weak: every rank owns a different rotation of the same seeded set (independent shards)
    k = (rank * 131) % max(len(files), 1)
    ids = list(range(k, len(files))) + list(range(k))
    return (files[k:] + files[:k], ids) if with_ids else files[k:] + files[:k]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:      # region shorter than the sampling period: use the nearest samples
            for ts, line in self.rows[-3:]:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1])); mx = float(f[2])
                except (ValueError, IndexError):
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU baseline: the reference compiled from its own sources (oracle/_ref), all host cores
# ---------------------------------------------------------------------------------------------
def _ref_worker(jpg: bytes) -> float:
    from oracle import refbind
    t = time.perf_counter()
    r = refbind.decode(jpg, mode=1, variant="hd", want_planes=False)
    assert r["rc"] == 0
    return time.perf_counter() - t


def _ref_file_worker(paths) -> float:
    """The reference's ConvertJpgFile sequence for one file (openjpg.cpp:593-684): read, parse + decode, WriteBMP24
    -- the reference's own code for every step (oracle/_ref), with heap buffers instead of the 105 KB stack
    buffer and restarts counted in MCUs by the harness (mode 1: the reference's own restart handling is
    broken, SURVEY.md 8c), exactly as in the cpu_baseline."""
    from oracle import refbind
    src, dst = paths
    t = time.perf_counter()
    jpg = open(src, "rb").read()
    r = refbind.decode(jpg, mode=1, variant="hd", want_planes=False)
    assert r["rc"] == 0
    refbind.write_bmp24(dst, r["rgb"])
    return time.perf_counter() - t


def _port_worker(jpg: bytes) -> float:
    from oracle import port
    t = time.perf_counter()
    r = port.decode(jpg, want_planes=False, want_coef=False)
    assert r["rc"] == 0
    return time.perf_counter() - t


class CpuReference:
    """The reference's CPU implementation of the path on a bounded sample: `per_core` images per
    host core, one process per core (the reference is single-threaded but re-entrant per process)."""

    def __init__(self, files: list[bytes], per_core: int = 1):
        from concurrent.futures import ProcessPoolExecutor
        from oracle import refbind
        self.cores = os.cpu_count() or 1
        self.kind = "reference" if refbind.available("hd") else "port"
        self.fn = _ref_worker if self.kind == "reference" else _port_worker
        n = min(len(files), self.cores * per_core)
        self.sample = files[:n]
        import multiprocessing as mp
        self.pool = ProcessPoolExecutor(max_workers=self.cores, mp_context=mp.get_context("spawn"))
        list(self.pool.map(self.fn, self.sample[: self.cores]))      # fork + load the .so before timing

    def step(self) -> float:
        t = time.perf_counter()
        list(self.pool.map(self.fn, self.sample))
        return time.perf_counter() - t

    def describe(self) -> str:
        return (f"{len(self.sample)} of the same 1920x1080 4:2:0 Ri=8 images per step, one process per core "
                f"({'reference sources compiled -O2 by oracle/build_ref.sh' if self.kind == 'reference' else 'oracle/jpeg_oracle.c port'})")

    def close(self):
        self.pool.shutdown()


def run_reference(args, rank, world):
    if rank != 0:
        return
    files = load_images(args.images or WORKLOADS["c2"]["n"], 0, 1)
    ref = CpuReference(files, per_core=1)
    for _ in range(args.warmup):
        ref.step()
    t = 0.0
    for _ in range(args.steps):
        t += ref.step()
    mp = len(ref.sample) * W * H / 1e6 * args.steps
    value = mp / t
    line = {"metric": "decoded_MP_per_s", "value": round(value, 3), "unit": "MP/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(1e3 * t / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"batch of synthetic {W}x{H} 4:2:0 baseline JPEGs, q85, restart interval 8 MCUs "
                                   f"(BASELINE.json configs[1]); CPU arm decodes a bounded sample per step"},
            "cpu_baseline": {"value": round(value, 3), "unit": "MP/s", "cores": ref.cores, "kind": ref.kind,
                             "sample": ref.describe()},
            "e2e": {"value": round(value, 3), "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    ref.close()
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# sub-records measured AFTER the timed headline (never inside it)
# ---------------------------------------------------------------------------------------------
def single_image_record(hjd, local_rank):
    """Config 1 through the reference-named single-image calls (DecodeJpgFileData loadjpg.h:186, ConvertJpgFile
    openjpg.cpp:593): wall-clock latency per call after the first.  The image is a synthetic stand-in of
    data/Lenna.jpg's shape (512x512 4:2:0, no restart markers: kernel 1b), since the reference's own file is
    not on the GPU box; tests/test_gpu_parity.py::test_lenna_config1 checks the real one where it exists."""
    import statistics
    from tools.gen_jpegs import encode_jpeg, synth_rgb
    jpg = encode_jpeg(synth_rgb(512, 512, 1), 92, "4:2:0", 0)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    src, dst = os.path.join(base, f"hjd_c1_{os.getpid()}.jpg"), os.path.join(base, f"hjd_c1_{os.getpid()}.bmp")
    with open(src, "wb") as fh:
        fh.write(jpg)
    try:
        hjd.lib().hjd_set_default_device(local_rank)
        for _ in range(5):
            hjd.DecodeJpgFileData(jpg)
            assert hjd.ConvertJpgFile(src, dst) == 1
        td, tc = [], []
        for _ in range(40):
            t = time.perf_counter(); hjd.DecodeJpgFileData(jpg); td.append(time.perf_counter() - t)
            t = time.perf_counter(); hjd.ConvertJpgFile(src, dst); tc.append(time.perf_counter() - t)
        return {"workload": f"one synthetic 512x512 4:2:0 baseline JPEG, {len(jpg)} bytes, no restart markers (the shape of configs[0]'s data/Lenna.jpg)",
                "DecodeJpgFileData_ms": round(1e3 * statistics.median(td), 3),
                "ConvertJpgFile_ms": round(1e3 * statistics.median(tc), 3), "calls": 40}
    finally:
        for p in (src, dst):
            if os.path.exists(p):
                os.remove(p)


def file_to_bmp_record(hjd, files, local_rank, rank, n_images=512, with_reference=False):
    """SURVEY.md 8(f) rank 3: .jpg files on disk -> .bmp files on disk through hjd_convert_jpg_files_multi
    (readers -> chunked GPU decodes in BMP layout -> writers), on a tmpfs so that the number is the
    pipeline's, not a disk's.  One file is checked against the oracle's WriteBMP24 bytes."""
    import shutil
    import numpy as np
    from oracle import port
    base = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    n = min(n_images, len(files))
    need = n * (W * H * 3 + 54) + sum(len(f) for f in files[:n])
    free = shutil.disk_usage(base).free
    if free < 2 * need:
        n = max(8, int(n * free / (2.5 * need)))
    root = os.path.join(base, f"hjd_f2b_{os.getpid()}")
    os.makedirs(root, exist_ok=True)
    try:
        ins, outs = [], []
        for i in range(n):
            p = os.path.join(root, f"{i:05d}.jpg")
            with open(p, "wb") as fh:
                fh.write(files[i])
            ins.append(p)
            outs.append(os.path.join(root, f"{i:05d}.bmp"))
        hjd.ConvertJpgFiles(ins[:8], outs[:8], device=local_rank)               # warm-up: contexts, page cache
        t = time.perf_counter()
        ok = hjd.ConvertJpgFiles(ins, outs, device=local_rank)
        t = time.perf_counter() - t
        assert all(ok), "file -> bmp conversion failed"
        o = port.decode(files[0], want_planes=False, want_coef=False)
        same = open(outs[0], "rb").read() == port.bmp24_bytes(o["rgb"])
        # the same pipeline with every output path = /dev/null: everything but the file system's write rate
        t_null = time.perf_counter()
        ok_null = hjd.ConvertJpgFiles(ins, ["/dev/null"] * n, device=local_rank)
        t_null = time.perf_counter() - t_null
        rec = {"images": n, "images_per_s": round(n / t, 1), "MP_per_s": round(n * W * H / 1e6 / t, 1),
               "bmp_GB_per_s": round(n * (W * H * 3 + 54) / t / 1e9, 2), "where": base,
               "images_per_s_to_dev_null": round(n / t_null, 1) if all(ok_null) else None,
               "bmp_bytes_identical_to_WriteBMP24": bool(same),
               "how": "hjd_convert_jpg_files_multi: file readers -> chunks of 32 images decoded with HJD_FLAG_BMP_OUT "
                      "-> writer threads; wall clock from the first fopen to the last fclose"}
        if with_reference:
            from concurrent.futures import ProcessPoolExecutor
            import multiprocessing as mp
            from oracle import refbind
            if refbind.available("hd"):
                cores = os.cpu_count() or 1
                m = min(n, cores)
                with ProcessPoolExecutor(max_workers=cores, mp_context=mp.get_context("spawn")) as ex:
                    pairs = [(ins[i], outs[i] + ".ref.bmp") for i in range(m)]
                    list(ex.map(_ref_file_worker, pairs[:cores]))            # load the .so before timing
                    t0 = time.perf_counter()
                    list(ex.map(_ref_file_worker, pairs))
                    t0 = time.perf_counter() - t0
                rec["reference_ConvertJpgFile"] = {"images_per_s": round(m / t0, 3), "cores": cores, "images": m,
                                                   "kind": "reference (oracle/_ref: its own parser, block decode and WriteBMP24; restarts counted by the harness)"}
                rec["reference_bmp_identical"] = open(pairs[0][1], "rb").read() == open(outs[0], "rb").read()
        return rec
    finally:
        shutil.rmtree(root, ignore_errors=True)


def dump_outputs(dec, out_dir):
    """What the last decode left for its caller, as float32 .npy files: every image's status and size, and its RGB at
    a fixed, seeded sample of pixel positions (the same positions for the same batch, whichever build decodes it)."""
    import numpy as np
    n = dec.num_images
    hw = np.array([(dec.info(i).height, dec.info(i).width) for i in range(n)], dtype=np.int64).reshape(n, 2)
    s = max(DUMP_PIXELS // max(n, 1), 1)
    u = np.random.default_rng(0).random((n, s))
    rgb = np.zeros((n, s, 3), dtype=np.float32)
    for i in range(n):
        h, w = (int(v) for v in hw[i])
        if h * w:
            pos = (u[i] * (h * w)).astype(np.int64)
            rgb[i] = dec.rgb(i).reshape(h * w, 3)[pos]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "status.npy"), dec.status().astype(np.float32))
    np.save(os.path.join(out_dir, "image_hw.npy"), hw.astype(np.float32))
    np.save(os.path.join(out_dir, "rgb.npy"), rgb)


def timed_resident(dec, steps, barrier):
    """K resident decodes bracketed by barriers; CUDA events on the launching stream.  Returns ms for the K steps
    and the stage times of the last one."""
    for _ in range(3):
        dec.decode()
    dec.sync()
    barrier()
    dec.mark(0)
    for _ in range(steps):
        dec.decode()
    dec.mark(1)
    dec.sync()
    barrier()
    return dec.elapsed_ms(0, 1), dec.timings()


def reduce_max_sum(dist, ms, sums):
    import torch
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    v = torch.tensor([float(x) for x in sums], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(v, op=dist.ReduceOp.SUM)
    return float(t.item()), [float(x) for x in v.tolist()]


def sub_record(hjd, dist, barrier, local_rank, rank, world, config, scaling, steps, peak):
    """One BASELINE.json workload, resident in HBM, K steps: whole-job MP/s, stage times, roofline fractions."""
    wl = WORKLOADS[config]
    files = load_images(wl["n"], rank, world, config, scaling)
    arena = hjd.PinnedArena(files)
    dec = hjd.BatchDecoder(local_rank)
    try:
        dec.upload_arena(arena)
        dec.sync()
        ms, t = timed_resident(dec, steps, barrier)
        st = dec.status()
        ok = bool((st == 0).all())
        alg = dec.scan_bytes + 3 * dec.pixels
        ms_max, (pix, scan, algs, imgs) = reduce_max_sum(dist, ms, [dec.pixels, dec.scan_bytes, alg, len(files)])
        stage = {k: round(t[k], 4) for k in ("scan_ms", "entropy_ms", "idct_ms", "color_ms")}
        dom = max(stage, key=stage.get)
        rec = {"workload": f"{int(imgs)} x {wl['desc']}", "scaling": scaling, "images_per_gpu_rank0": len(files),
               "steps": steps, "ms_per_step": round(ms_max / steps, 4),
               "MP_per_s": round(pix / 1e6 * steps / (ms_max / 1e3), 1),
               "compressed_GB_per_s": round(scan * steps / (ms_max / 1e3) / 1e9, 2),
               "stage_ms_rank0": stage, "status_ok": ok,
               "roofline": {"bound": "hbm", "kernel": dom.replace("_ms", ""),
                            "frac": round(alg / (max(stage[dom], 1e-6) / 1e3) / 1e9 / peak, 4),
                            "whole_step_frac": round(algs / (ms_max / steps / 1e3) / 1e9 / peak / world, 4),
                            "algorithmic_bytes_per_step": int(algs)}}
        if config in ("c4", "c2nr"):
            rec["selfsync_rounds"] = dec.selfsync_rounds
        return rec
    finally:
        dec.close()
        arena.close()


def parity_block(hjd, dist, dec, files, file_ids, rank, world, k):
    """Result check of the TIMED batch, outside the timed region.  Per rank: k images of its batch, spread over
    it, are (a) entropy-decoded by the oracle and compared coefficient for coefficient with what the GPU left
    in the slab, (b) for one of them, decoded in full by the oracle and compared pixel for pixel; (c) the sha256
    of every checked image's RGB is gathered, and rank 0 -- which holds every file -- decodes the same file
    ids itself and compares: rank r's image equals rank 0's decode of the same file."""
    import hashlib
    import numpy as np
    from oracle import port
    n = len(files)
    pick = sorted(set(int(round(j * (n - 1) / max(k - 1, 1))) for j in range(min(k, n))))
    coef_bad = blocks = rgb_bad = 0
    shas = []
    for j, i in enumerate(pick):
        o = port.decode(files[i], entropy_only=(j != 0), want_planes=False)
        got = dec.image_coefficients_direct(i)
        coef_bad += int((got != o["coef"]).any(axis=1).sum())
        blocks += got.shape[0]
        rgb = dec.rgb(i)
        if j == 0:
            rgb_bad += int((rgb != o["rgb"]).sum())
        shas.append((int(file_ids[i]), hashlib.sha256(rgb.tobytes()).hexdigest()))
    gathered = [shas]
    if dist is not None:
        gathered = [None] * world
        dist.all_gather_object(gathered, shas)
    cross_bad = cross = 0
    if rank == 0:
        want = {}
        todo = sorted({fid for g in gathered for fid, _ in g})
        all_files = load_images(WORKLOADS["c2"]["n"], 0, 1)
        with hjd.BatchDecoder(dec.device) as d2:
            d2.upload([all_files[fid] for fid in todo])
            d2.decode()
            for q, fid in enumerate(todo):
                want[fid] = hashlib.sha256(d2.rgb(q).tobytes()).hexdigest()
        for g in gathered:
            for fid, h in g:
                cross += 1
                cross_bad += int(want[fid] != h)
    import torch
    v = torch.tensor([float(len(pick)), float(blocks), float(coef_bad), float(rgb_bad)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(v, op=dist.ReduceOp.SUM)
    imgs, blocks, coef_bad, rgb_bad = (int(x) for x in v.tolist())
    return {"checker": "oracle/jpeg_oracle.c (restatement pinned to the reference, tests/test_oracle.py)",
            "images_checked": imgs, "coef_blocks_checked": blocks, "coef_block_mismatches": coef_bad,
            "rgb_full_compares": world, "rgb_sample_mismatches": rgb_bad,
            "cross_rank_sha_checked": cross, "cross_rank_sha_mismatches": cross_bad,
            "mismatches": coef_bad + rgb_bad + cross_bad}


# ---------------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import numpy as np
    import torch
    import hls_jpeg_decoder_b200 as hjd

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    wl = WORKLOADS[args.config]
    n_req = args.images or wl["n"]
    files, file_ids = load_images(n_req, rank, world, args.config, args.scaling, with_ids=True)
    n = len(files)
    arena = hjd.PinnedArena(files, device=local_rank)       # pinned pages from the NUMA node next to this GPU, if any
    dec = hjd.BatchDecoder(local_rank, int(os.environ.get("HJD_BENCH_FLAGS", "0")))     # experiments only: e.g. 128 = HJD_FLAG_TENSOR_CORE_IDCT
    dec.upload_arena(arena)
    dec.sync()
    pixels, scan_bytes = dec.pixels, dec.scan_bytes
    working_set = dec.coef_bytes + dec.rgb_bytes
    alg_bytes = scan_bytes + 3 * pixels                   # SURVEY.md 8(d): B_alg = scan bytes in + RGB out

    for _ in range(max(args.warmup, 3)):
        dec.decode()
    dec.sync()
    st = dec.status()
    assert (st == 0).all(), f"decode status: {st[st != 0][:8]}"

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    stage = {"scan_ms": 0.0, "entropy_ms": 0.0, "idct_ms": 0.0, "color_ms": 0.0}
    launches = 0
    barrier()
    t0 = time.time()
    per_step = args.steps <= 128             # one event per step boundary as long as the slots last
    dec.mark(0)
    for i in range(args.steps):
        dec.decode()
        if per_step and i + 1 < args.steps:
            dec.mark(2 + i)
    dec.mark(1)
    dec.sync()
    barrier()
    t1 = time.time()
    ms_total = dec.elapsed_ms(0, 1)
    step_ms = []
    if per_step:
        marks = [0] + [2 + i for i in range(args.steps - 1)] + [1]
        step_ms = sorted(dec.elapsed_ms(marks[i], marks[i + 1]) for i in range(args.steps))
    clocks = sampler.stop(t0, t1)
    # per-stage CUDA-event times of the LAST TIMED step (the HBM-resident decode runs on one stream, in
    # order, and records its stage boundaries on that stream at every step): the roofline's kernel
    # duration is measured inside the timed region, not in a separate run
    t = dec.timings()
    for k in stage:
        stage[k] = t[k]
    launches = t["launches"]
    idct_variant = dec.idct_variant          # which fused kernel(s) the timed decodes went through (read while the batch is alive)
    if args.dump_outputs and rank == 0:      # before the end-to-end leg decodes through the same handle again
        dump_outputs(dec, args.dump_outputs)

    t_ms = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(pixels), float(scan_bytes), float(alg_bytes), float(n), float(launches * args.steps)],
                       dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_max = float(t_ms.item())
    job_pixels, job_scan, job_alg, job_images, job_launches = (float(v) for v in tot.tolist())
    value = job_pixels / 1e6 * args.steps / (ms_max / 1e3)

    # end to end through the C ABI with host buffers (pinned in, pinned out), copies inside the timed region
    e2e = None
    if not args.no_e2e:
        need = hjd.rgb_slab_bytes(arena)
        out_ptr = hjd.lib().hjd_host_alloc_near(local_rank, need)
        if not out_ptr:
            raise RuntimeError("pinned output allocation failed")
        dec.set_overlap(1)
        dec.decode_host(arena, out_ptr, need, 0)           # warm-up (allocations)
        barrier()
        te = time.perf_counter()
        for _ in range(args.e2e_steps):
            _, st2 = dec.decode_host(arena, out_ptr, need, 0)
        barrier()
        te = time.perf_counter() - te
        assert (st2 == 0).all()
        t_e = torch.tensor([te], dtype=torch.float64, device="cuda")
        io = torch.tensor([float(arena.bytes), float(need)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
            dist.all_reduce(io, op=dist.ReduceOp.SUM)          # whole job, like the value
        e2e = {"value": round(job_pixels / 1e6 * args.e2e_steps / float(t_e.item()), 1), "unit": "MP/s",
               "h2d_bytes_per_step": int(io[0].item()), "d2h_bytes_per_step": int(io[1].item()), "steps": args.e2e_steps}
        # the ceiling of this host link: the same bytes, the same pinned buffers, all ranks at once, NO kernels
        barrier()
        ms_up, ms_down = hjd.link_probe(local_rank, arena.ptr, arena.bytes, out_ptr, need, reps=max(args.e2e_steps, 2))
        barrier()
        t_l = torch.tensor([max(ms_up, ms_down)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t_l, op=dist.ReduceOp.MAX)
        t_link = float(t_l.item()) / 1e3
        e2e["link_ceiling"] = {"value": round(job_pixels / 1e6 / t_link, 1), "unit": "MP/s",
                               "d2h_GB_per_s": round(e2e["d2h_bytes_per_step"] / t_link / 1e9, 2),
                               "h2d_GB_per_s": round(e2e["h2d_bytes_per_step"] / t_link / 1e9, 2),
                               "numa_node_rank0": hjd.lib().hjd_device_numa_node(local_rank),
                               "how": "hjd_link_probe: per rank, this step's H2D and D2H bytes copied concurrently between the same "
                                      "pinned buffers and HBM with no kernel running, all ranks at once, max over ranks"}
        e2e["frac_of_link_ceiling"] = round(e2e["value"] / e2e["link_ceiling"]["value"], 4)
        hjd.lib().hjd_host_free(out_ptr)

    # sub-records after the timed regions: parity of the timed batch, then the other BASELINE.json configs
    extras = {}
    if not args.no_extras and args.config == "c2" and args.scaling == "weak":
        peak0 = measured_peak()[0]
        extras["parity"] = parity_block(hjd, dist, dec, files, file_ids, rank, world, args.parity_images)
        dec.close()
        arena.close()
        if rank == 0:
            extras["c1"] = single_image_record(hjd, local_rank)
            extras["file_to_bmp"] = file_to_bmp_record(hjd, files, local_rank, rank, with_reference=(world == 1 and not args.no_cpu_baseline))
        barrier()
        strong = sub_record(hjd, dist, barrier, local_rank, rank, world, "c2", "strong", args.extra_steps, peak0)
        # every rank of the weak headline decoded the whole 1024-image batch on one GPU: its step time is t(1)
        strong["efficiency_vs_1gpu"] = round((ms_max / args.steps) / (world * strong["ms_per_step"]), 4)
        strong["ms_per_step_1gpu"] = round(ms_max / args.steps, 4)
        extras["strong"] = strong
        extras["c4"] = sub_record(hjd, dist, barrier, local_rank, rank, world, "c4", "weak", args.extra_steps, peak0)
        extras["c5"] = sub_record(hjd, dist, barrier, local_rank, rank, world, "c5", "weak", args.extra_steps, peak0)
        dec = arena = None

    if rank == 0:
        peak, peak_src = measured_peak()
        dom = max(stage, key=stage.get)
        dom_ms = stage[dom]
        achieved = alg_bytes / (dom_ms / 1e3) / 1e9
        traffic = None
        try:   # DRAM bytes per launch of that kernel from the committed ncu capture, scaled to this batch
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_final_traffic.json")))
            if args.config == "c2":
                traffic = int(tj["dram_bytes_per_launch"][dom.replace("_ms", "")] * n / tj["images"])
        except Exception:
            traffic = None
        whole = alg_bytes / (ms_max / args.steps / 1e3) / 1e9
        line = {"metric": "decoded_MP_per_s", "value": round(value, 1), "unit": "MP/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_max / args.steps, 4),
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"{int(job_images)} x {wl['desc']}; inputs resident in HBM",
                           "images_per_gpu": n, "scan_bytes_per_image": scan_bytes // max(n, 1),
                           "l2_policy": f"per-step working set (coefficient + RGB slabs, {working_set / 1e9:.2f} GB on rank 0) "
                                        "against a 126 MB L2; every step rewrites all of it",
                           "parallelism": f"{world} independent shards ({args.scaling} scaling), no collective",
                           "idct_kernel": {1: "tensor cores: tcgen05.mma, FP16 x FP16 -> FP32 with exact integer accumulation (csrc/mcu_tc.cuh)",
                                           2: "CUDA cores: FP32 FMA chains (csrc/kernels.cu)",
                                           3: "tensor cores and CUDA cores, chosen per chunk"}.get(idct_variant, "none")},
                "compressed_GB_per_s": round(job_scan * args.steps / (ms_max / 1e3) / 1e9, 2),
                "stage_ms": {k: round(v, 4) for k, v in stage.items()},
                "roofline": {"bound": "hbm", "kernel": dom.replace("_ms", ""), "achieved": round(achieved, 1),
                             "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
                             "traffic_source": "profiles/r2_final_traffic.json (ncu --set full, per launch)" if traffic else None,
                             "peak_source": peak_src, "algorithmic_bytes_per_step": int(alg_bytes),
                             "whole_step_frac": round(whole / peak, 4)},
                "clocks": clocks, "gpu_launches": int(job_launches)}
        if step_ms:     # rank 0's own steps, CUDA events between consecutive steps (SURVEY.md 8d: best and median)
            line["ms_per_step_best"] = round(step_ms[0], 4)
            line["ms_per_step_median"] = round(step_ms[len(step_ms) // 2], 4)
        if e2e:
            line["e2e"] = e2e
        line.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            ref = CpuReference(load_images(WORKLOADS["c2"]["n"], 0, 1) if args.config != "c2" else files, per_core=1)
            ref.step()
            t = ref.step()
            line["cpu_baseline"] = {"value": round(len(ref.sample) * W * H / 1e6 / t, 3), "unit": "MP/s",
                                    "cores": ref.cores, "kind": ref.kind, "sample": ref.describe()}
            ref.close()
        print(json.dumps(line), flush=True)
    if dec is not None:
        dec.close()
        arena.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank, local_rank, world = rank_env()
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
