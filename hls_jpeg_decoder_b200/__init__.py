"""hls_jpeg_decoder_b200 -- B200-native baseline-JPEG decode path behind the entry points of
harutel/hls-jpeg-decoder.

This package is a thin ctypes binding of ``libhjd.so`` (include/hjd.h): host C++ parses the
JPEG headers and builds the tables, hand-written sm_100a CUDA kernels do all decoding.  There
is no CPU fallback: if the shared library or a CUDA device is missing, calls raise.

Reference-shaped API (same names, argument meaning and 1/0 return convention as the reference):

    ConvertJpgFile(jpg_in, bmp_out) -> int              openjpg.cpp:593
    DecodeJpgFileData(buf) -> (rgb[h, w, 3] uint8, w, h) loadjpg.h:186
    JpegGetImageSize(buf) -> (w, h)                     loadjpg.h:183
    WriteBMP24(path, w, h, rgb)                         openjpg.cpp:504

Batch API (the JpegDecodeHW replacement for N independent images): :class:`BatchDecoder`.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint, c_uint8, c_uint32, c_uint64, c_void_p

import numpy as np

__all__ = ["probe", "MultiDecoder", "shard_range_c", "ConvertJpgFile", "ConvertJpgFiles", "DecodeJpgFileData", "JpegGetImageSize", "WriteBMP24", "encode_bmp24",
           "BatchDecoder", "HjdError", "lib", "build", "LIB_PATH",
           "FLAG_KEEP_PLANES", "FLAG_HOST_SCAN", "FLAG_NO_SELFSYNC", "FLAG_FUSED_MCU", "FLAG_BMP_OUT", "FLAG_TENSOR_CORE_IDCT", "FLAG_CUDA_CORE_IDCT", "FLAG_MULTI_SCAN", "FLAG_SCALE_1_2",
           "FLAG_SCALE_1_4", "FLAG_SCALE_1_8", "FLAG_GRAY_OUT", "FLAG_EXIF_ORIENT", "scans", "orientation", "idct_matrix", "idct_tables"]

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HJD_LIB_PATH") or os.path.join(_HERE, "libhjd.so")   # override: tuning builds only
INCLUDE_PATH = os.path.join(os.path.dirname(_HERE), "include", "hjd.h")

FLAG_KEEP_PLANES = 1
FLAG_HOST_SCAN = 2
FLAG_NO_SELFSYNC = 8
FLAG_FUSED_MCU = 16
FLAG_BMP_OUT = 32
FLAG_TENSOR_CORE_IDCT = 128  # always the fused kernel with the IDCT's fast tier as tcgen05.mma
FLAG_CUDA_CORE_IDCT = 64     # always the fused kernel with the fast tier as FP32 FMA chains (default: chosen per chunk)
FLAG_MULTI_SCAN = 256        # also decode progressive and non-interleaved files (each exactly like its baseline twin)
FLAG_SCALE_1_2 = 1 << 9      # decode to ceil(W/2) x ceil(H/2) in the DCT domain (include/hjd.h; not with KEEP_PLANES,
FLAG_SCALE_1_4 = 2 << 9      # BMP_OUT, TENSOR_CORE_IDCT or CUDA_CORE_IDCT)
FLAG_SCALE_1_8 = 3 << 9      # 1/8: a block is its DC alone; with MULTI_SCAN the AC scans are not read
FLAG_GRAY_OUT = 1 << 11      # one byte per pixel: the decoded Y component (BatchDecoder.gray; include/hjd.h; not with
                             # KEEP_PLANES, BMP_OUT, TENSOR_CORE_IDCT or CUDA_CORE_IDCT)
FLAG_EXIF_ORIENT = 1 << 12   # apply each file's EXIF orientation to its output (out_size swaps for 5-8; include/hjd.h; not
                             # with BMP_OUT)

IMG_WARN_BAD_CODE, IMG_WARN_COEF_RANGE, IMG_WARN_OVERRUN, IMG_WARN_RESTART = 1, 2, 4, 8


class HjdError(RuntimeError):
    pass


class ImageInfo(ctypes.Structure):
    _fields_ = [("width", c_uint32), ("height", c_uint32), ("ncomp", c_uint8), ("hf", c_uint8), ("vf", c_uint8),
                ("blocks_per_mcu", c_uint8), ("mcus_x", c_uint32), ("mcus_y", c_uint32),
                ("restart_interval", c_uint32), ("n_intervals", c_uint32), ("scan_bytes", c_uint32),
                ("block_base", c_uint64), ("n_blocks", c_uint64), ("rgb_offset", c_uint64),
                ("y_offset", c_uint64), ("cb_offset", c_uint64), ("cr_offset", c_uint64),
                ("y_pitch", c_uint32), ("c_pitch", c_uint32), ("status", c_int32)]


class ScanInfo(ctypes.Structure):
    _fields_ = [("ncomp", c_uint8), ("comp", c_uint8 * 3), ("ss", c_uint8), ("se", c_uint8), ("ah", c_uint8),
                ("al", c_uint8), ("level", c_uint8), ("pad", c_uint8 * 3), ("restart_interval", c_uint32),
                ("bytes", c_uint32)]


class Timings(ctypes.Structure):
    _fields_ = [("scan_ms", c_float), ("entropy_ms", c_float), ("idct_ms", c_float), ("color_ms", c_float),
                ("total_ms", c_float), ("launches", c_int)]


def build(force: bool = False) -> str:
    """Compile libhjd.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc")] + (["-B"] if force else [])
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None

_SIGS = {
    "hjd_version": (c_int, []),
    "hjd_last_error": (c_char_p, []),
    "hjd_device_count": (c_int, []),
    "hjd_convert_jpg_file": (c_int, [c_char_p, c_char_p]),
    "hjd_decode_jpg_file_data": (c_int, [c_void_p, c_int, POINTER(c_void_p), POINTER(c_uint), POINTER(c_uint)]),
    "hjd_free": (None, [c_void_p]),
    "hjd_get_image_size": (c_int, [c_void_p, c_int, POINTER(c_uint), POINTER(c_uint)]),
    "hjd_write_bmp24": (c_int, [c_char_p, c_uint, c_uint, c_void_p]),
    "hjd_encode_bmp24": (c_size_t, [c_uint, c_uint, c_void_p, c_void_p]),
    "hjd_convert_jpg_files": (c_int, [POINTER(c_char_p), POINTER(c_char_p), c_int, c_int, c_int, POINTER(c_int)]),
    "hjd_batch_create": (c_void_p, [c_int, c_uint]),
    "hjd_batch_destroy": (None, [c_void_p]),
    "hjd_batch_set_stream": (c_int, [c_void_p, c_void_p]),
    "hjd_batch_upload": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_int64), c_int]),
    "hjd_batch_upload_arena": (c_int, [c_void_p, c_void_p, POINTER(c_int64), POINTER(c_int64), c_int]),
    "hjd_batch_decode": (c_int, [c_void_p]),
    "hjd_batch_sync": (c_int, [c_void_p]),
    "hjd_batch_set_overlap": (c_int, [c_void_p, c_int]),
    "hjd_batch_set_selfsync_range": (c_int, [c_void_p, c_int]),
    "hjd_batch_num_images": (c_int, [c_void_p]),
    "hjd_batch_selfsync_rounds": (c_int, [c_void_p]),
    "hjd_batch_idct_variant": (c_int, [c_void_p]),
    "hjd_batch_get_info": (c_int, [c_void_p, c_int, POINTER(ImageInfo)]),
    "hjd_batch_get_status": (c_int, [c_void_p, c_void_p]),
    "hjd_batch_get_timings": (c_int, [c_void_p, POINTER(Timings)]),
    "hjd_batch_mark": (c_int, [c_void_p, c_int]),
    "hjd_batch_elapsed_ms": (c_float, [c_void_p, c_int, c_int]),
    "hjd_batch_rgb_bytes": (c_uint64, [c_void_p]),
    "hjd_batch_coef_bytes": (c_uint64, [c_void_p]),
    "hjd_batch_plane_bytes": (c_uint64, [c_void_p]),
    "hjd_batch_scan_bytes": (c_uint64, [c_void_p]),
    "hjd_batch_pixels": (c_uint64, [c_void_p]),
    "hjd_batch_device_rgb": (c_void_p, [c_void_p]),
    "hjd_batch_device_coef": (c_void_p, [c_void_p]),
    "hjd_batch_device_planes": (c_void_p, [c_void_p]),
    "hjd_batch_download_rgb": (c_int, [c_void_p, c_void_p]),
    "hjd_batch_download_image": (c_int, [c_void_p, c_int, c_void_p]),
    "hjd_batch_download_coef": (c_int, [c_void_p, c_void_p]),
    "hjd_batch_download_planes": (c_int, [c_void_p, c_void_p]),
    "hjd_batch_download_image_coef": (c_int, [c_void_p, c_int, c_void_p]),
    "hjd_batch_bmp_bytes": (c_uint64, [c_void_p, c_int]),
    "hjd_batch_download_bmp": (c_int, [c_void_p, c_int, c_void_p]),
    "hjd_out_slab_bytes": (c_uint64, [c_void_p, POINTER(c_int64), POINTER(c_int64), c_int, c_uint]),
    "hjd_batch_decode_host": (c_int, [c_void_p, c_void_p, POINTER(c_int64), POINTER(c_int64), c_int, c_void_p,
                                      c_uint64, POINTER(c_uint64), c_void_p, c_int]),
    "hjd_rgb_slab_bytes": (c_uint64, [c_void_p, POINTER(c_int64), POINTER(c_int64), c_int]),
    "hjd_host_alloc": (c_void_p, [c_size_t]),
    "hjd_host_free": (None, [c_void_p]),
    "hjd_host_alloc_near": (c_void_p, [c_int, c_size_t]),
    "hjd_device_numa_node": (c_int, [c_int]),
    "hjd_link_probe": (c_int, [c_int, c_void_p, c_size_t, c_void_p, c_size_t, c_int, POINTER(c_float), POINTER(c_float)]),
    "hjd_get_idct_tables": (None, [c_void_p, c_void_p]),
    "hjd_get_idct_matrix": (None, [c_void_p]),
    "hjd_decode_jpg_file_data_alloc": (c_int, [c_void_p, c_int, c_void_p, POINTER(c_void_p), POINTER(c_uint), POINTER(c_uint)]),
    "hjd_set_default_device": (c_int, [c_int]),
    "hjd_convert_jpg_files_multi": (c_int, [POINTER(c_char_p), POINTER(c_char_p), c_int, POINTER(c_int), c_int, c_int, c_int, POINTER(c_int)]),
    "hjd_shard_range": (c_int, [POINTER(c_int64), c_int, c_int, c_int, POINTER(c_int), POINTER(c_int)]),
    "hjd_multi_create": (c_void_p, [POINTER(c_int), c_int, c_uint]),
    "hjd_multi_destroy": (None, [c_void_p]),
    "hjd_multi_num_devices": (c_int, [c_void_p]),
    "hjd_multi_batch": (c_void_p, [c_void_p, c_int]),
    "hjd_multi_last_error": (c_char_p, [c_void_p]),
    "hjd_multi_out_slab_bytes": (c_uint64, [c_void_p, c_void_p, POINTER(c_int64), POINTER(c_int64), c_int]),
    "hjd_multi_decode_host": (c_int, [c_void_p, c_void_p, POINTER(c_int64), POINTER(c_int64), c_int, c_void_p, c_uint64,
                                      POINTER(c_uint64), c_void_p]),
    "hjd_probe_jpeg": (c_int, [c_void_p, c_int64, POINTER(ImageInfo)]),
    "hjd_probe_jpeg_flags": (c_int, [c_void_p, c_int64, c_uint, POINTER(ImageInfo)]),
    "hjd_probe_jpeg_scans": (c_int, [c_void_p, c_int64, POINTER(ScanInfo), c_int]),
    "hjd_batch_num_scans": (c_int, [c_void_p, c_int]),
    "hjd_batch_get_out_size": (c_int, [c_void_p, c_int, POINTER(c_uint32), POINTER(c_uint32)]),
    "hjd_batch_get_orientation": (c_int, [c_void_p, c_int]),
    "hjd_probe_jpeg_orientation": (c_int, [c_void_p, c_int64]),
    "hjd_huff_lookup_probe": (c_uint32, [c_void_p, c_void_p, c_int, c_int, c_uint32]),
}


def lib() -> ctypes.CDLL:
    """The loaded C-ABI library.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HjdError(f"{LIB_PATH} is missing: build it with hls_jpeg_decoder_b200.build() "
                           "(nvcc, sm_100a); this package has no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def _err() -> str:
    return lib().hjd_last_error().decode(errors="replace")


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise HjdError(f"{what} failed ({rc}): {_err()}")


# ---------------------------------------------------------------------------------------------
# reference-shaped entry points
# ---------------------------------------------------------------------------------------------
def ConvertJpgFile(szJpgFileInName: str, szBmpFileOutName: str) -> int:
    """openjpg.cpp:593 -- load a .jpg, decode it on the GPU, write a 24-bit .bmp.  1 = ok, 0 = failure."""
    return int(lib().hjd_convert_jpg_file(os.fsencode(szJpgFileInName), os.fsencode(szBmpFileOutName)))


def ConvertJpgFiles(jpg_in: list[str], bmp_out: list[str], device: int = 0, threads: int = 0,
                    devices: list[int] | None = None, chunk_images: int = 0) -> list[int]:
    """ConvertJpgFile at batch scale: a pipeline of parallel file readers, chunked GPU decodes that write
    the BMP file layout, and parallel file writers, on one device or a list of them.
    Returns the per-file 1/0 flags."""
    n = len(jpg_in)
    assert len(bmp_out) == n
    a = (c_char_p * n)(*[os.fsencode(p) for p in jpg_in])
    b = (c_char_p * n)(*[os.fsencode(p) for p in bmp_out])
    ok = (c_int * n)()
    devs = list(devices) if devices else [device]
    lib().hjd_convert_jpg_files_multi(a, b, n, (c_int * len(devs))(*devs), len(devs), threads, chunk_images, ok)
    return list(ok)


def DecodeJpgFileData(buf: bytes):
    """loadjpg.h:186 -- whole .jpg file in memory -> (rgb[h, w, 3] uint8, width, height)."""
    data = np.frombuffer(buf, dtype=np.uint8)
    out, w, h = c_void_p(), c_uint(), c_uint()
    ok = lib().hjd_decode_jpg_file_data(data.ctypes.data, data.size, ctypes.byref(out), ctypes.byref(w), ctypes.byref(h))
    if not ok:
        raise HjdError(f"DecodeJpgFileData failed: {_err()}")
    try:
        n = w.value * h.value * 3
        rgb = np.ctypeslib.as_array(ctypes.cast(out, POINTER(c_uint8)), shape=(n,)).copy().reshape(h.value, w.value, 3)
    finally:
        lib().hjd_free(out)
    return rgb, w.value, h.value


def JpegGetImageSize(buf: bytes):
    """loadjpg.h:183 -- (width, height) from the file header."""
    data = np.frombuffer(buf, dtype=np.uint8)
    w, h = c_uint(), c_uint()
    if not lib().hjd_get_image_size(data.ctypes.data, data.size, ctypes.byref(w), ctypes.byref(h)):
        raise HjdError(f"JpegGetImageSize failed: {_err()}")
    return w.value, h.value


def probe(buf: bytes, flags: int = 0):
    """Header parse only (no GPU): (status, ImageInfo) -- the per-image status a batch created with `flags` would report."""
    data = np.frombuffer(buf, dtype=np.uint8)
    o = ImageInfo()
    st = lib().hjd_probe_jpeg_flags(data.ctypes.data if data.size else None, data.size, flags, ctypes.byref(o))
    return int(st), o


def scans(buf: bytes) -> list[dict]:
    """The scans a FLAG_MULTI_SCAN batch decodes the file from (no GPU): one dict per scan with ncomp, comp (frame
    component indices), ss, se, ah, al, level, restart_interval, bytes.  Raises HjdError for an undecodable file."""
    data = np.frombuffer(buf, dtype=np.uint8)
    ptr = data.ctypes.data if data.size else None
    n = lib().hjd_probe_jpeg_scans(ptr, data.size, None, 0)
    if n < 0:
        raise HjdError(f"not a decodable JPEG (status {n})")
    out = (ScanInfo * max(n, 1))()
    lib().hjd_probe_jpeg_scans(ptr, data.size, out, n)
    return [dict(ncomp=s.ncomp, comp=list(s.comp[:s.ncomp]), ss=s.ss, se=s.se, ah=s.ah, al=s.al, level=s.level,
                 restart_interval=s.restart_interval, bytes=s.bytes) for s in out[:n]]


def orientation(buf: bytes) -> int:
    """The EXIF orientation (1..8) the file states, as FLAG_EXIF_ORIENT applies it (header parse only, no GPU); 1 when
    the file has none or a malformed one.  Raises HjdError when the buffer does not start with SOI."""
    data = np.frombuffer(buf, dtype=np.uint8)
    o = lib().hjd_probe_jpeg_orientation(data.ctypes.data if data.size else None, data.size)
    if o < 1:
        raise HjdError(f"not a JPEG (status {o})")
    return int(o)


def WriteBMP24(szBmpFileName: str, Width: int, Height: int, RGB) -> None:
    """openjpg.cpp:504 -- 24-bit bottom-up BGR BMP, byte-identical to the reference's writer."""
    rgb = np.ascontiguousarray(RGB, dtype=np.uint8)
    if rgb.size != Width * Height * 3:
        raise ValueError("RGB buffer does not match Width*Height*3")
    if not lib().hjd_write_bmp24(os.fsencode(szBmpFileName), Width, Height, rgb.ctypes.data):
        raise HjdError(f"WriteBMP24 failed: {_err()}")


def encode_bmp24(rgb: np.ndarray) -> bytes:
    h, w, _ = rgb.shape
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    n = lib().hjd_encode_bmp24(w, h, rgb.ctypes.data, None)
    out = np.empty(n, dtype=np.uint8)
    lib().hjd_encode_bmp24(w, h, rgb.ctypes.data, out.ctypes.data)
    return out.tobytes()


# ---------------------------------------------------------------------------------------------
# batch API
# ---------------------------------------------------------------------------------------------
class PinnedArena:
    """Files packed back to back (16-byte aligned) in pinned host memory."""

    def __init__(self, files: list[bytes], device: int | None = None):
        L = lib()
        self.n = len(files)
        self.sizes = (c_int64 * self.n)(*[len(f) for f in files])
        offs, o = [], 0
        for f in files:
            offs.append(o)
            o += (len(f) + 15) // 16 * 16
        self.offsets = (c_int64 * self.n)(*offs)
        self.bytes = max(o, 16)
        self.ptr = L.hjd_host_alloc(self.bytes) if device is None else L.hjd_host_alloc_near(device, self.bytes)
        if not self.ptr:
            raise HjdError(f"pinned allocation of {self.bytes} bytes failed: {_err()}")
        self.view = np.ctypeslib.as_array(ctypes.cast(self.ptr, POINTER(c_uint8)), shape=(self.bytes,))
        for f, off in zip(files, offs):
            self.view[off:off + len(f)] = np.frombuffer(f, dtype=np.uint8)

    def close(self):
        if self.ptr:
            self.view = None
            lib().hjd_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchDecoder:
    """One per GPU.  upload() parses + copies N files to HBM, decode() launches the kernels,
    results stay in HBM until downloaded."""

    def __init__(self, device: int = 0, flags: int = 0):
        self._h = lib().hjd_batch_create(device, flags)
        if not self._h:
            raise HjdError(f"hjd_batch_create failed: {_err()}")
        self.device = device
        self.flags = flags
        self._keep = None

    def close(self):
        if self._h:
            lib().hjd_batch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- input -------------------------------------------------------------------------------
    def upload(self, files: list[bytes]) -> None:
        n = len(files)
        arrs = [np.frombuffer(f, dtype=np.uint8) for f in files]
        ptrs = (c_void_p * n)(*[a.ctypes.data for a in arrs])
        sizes = (c_int64 * n)(*[a.size for a in arrs])
        self._keep = arrs
        _check(lib().hjd_batch_upload(self._h, ptrs, sizes, n), "hjd_batch_upload")
        _check(lib().hjd_batch_sync(self._h), "hjd_batch_sync")

    def upload_arena(self, arena: PinnedArena, first: int = 0, count: int | None = None) -> None:
        count = arena.n - first if count is None else count
        offs = ctypes.cast(ctypes.byref(arena.offsets, first * 8), POINTER(c_int64))
        sizes = ctypes.cast(ctypes.byref(arena.sizes, first * 8), POINTER(c_int64))
        self._keep = arena
        _check(lib().hjd_batch_upload_arena(self._h, arena.ptr, offs, sizes, count), "hjd_batch_upload_arena")

    # -- compute -----------------------------------------------------------------------------
    def decode(self) -> None:
        _check(lib().hjd_batch_decode(self._h), "hjd_batch_decode")

    def sync(self) -> None:
        _check(lib().hjd_batch_sync(self._h), "hjd_batch_sync")

    def set_overlap(self, on) -> None:
        """Chunked multi-stream execution: 0/False = one stream (per-stage timings valid), 1/True =
        default chunking, n > 1 = target blocks per chunk.  Takes effect at the next upload."""
        _check(lib().hjd_batch_set_overlap(self._h, int(on)), "hjd_batch_set_overlap")

    def set_selfsync_range(self, rng: int) -> None:
        """Sub-sequences per warp in the synchronisation rounds of the restart-free path (0 = automatic).
        Results do not depend on it; takes effect at the next upload."""
        _check(lib().hjd_batch_set_selfsync_range(self._h, int(rng)), "hjd_batch_set_selfsync_range")

    def mark(self, slot: int) -> None:
        _check(lib().hjd_batch_mark(self._h, slot), "hjd_batch_mark")

    def elapsed_ms(self, a: int, b: int) -> float:
        ms = lib().hjd_batch_elapsed_ms(self._h, a, b)
        if ms < 0:
            raise HjdError(f"hjd_batch_elapsed_ms failed: {_err()}")
        return float(ms)

    def timings(self) -> dict:
        t = Timings()
        _check(lib().hjd_batch_get_timings(self._h, ctypes.byref(t)), "hjd_batch_get_timings")
        return {k: getattr(t, k) for k, _ in Timings._fields_}

    # -- results -----------------------------------------------------------------------------
    @property
    def selfsync_rounds(self) -> int:
        return lib().hjd_batch_selfsync_rounds(self._h)

    @property
    def idct_variant(self) -> int:
        """bit 0: chunks of the last decode went through the tensor-core fused kernel; bit 1: through the CUDA-core one;
        bit 2: through the scaled kernel (FLAG_SCALE_*); bit 3: through a luma-only kernel (FLAG_GRAY_OUT)"""
        return lib().hjd_batch_idct_variant(self._h)

    @property
    def num_images(self) -> int:
        return lib().hjd_batch_num_images(self._h)

    def num_scans(self, i: int) -> int:
        """Scans image i of the last upload is decoded from (1: single-scan baseline, 0: not decodable)."""
        n = lib().hjd_batch_num_scans(self._h, i)
        if n < 0:
            raise HjdError(f"hjd_batch_num_scans failed: {_err()}")
        return n

    def info(self, i: int) -> ImageInfo:
        o = ImageInfo()
        _check(lib().hjd_batch_get_info(self._h, i, ctypes.byref(o)), "hjd_batch_get_info")
        return o

    def status(self) -> np.ndarray:
        out = np.zeros(max(self.num_images, 1), dtype=np.int32)
        _check(lib().hjd_batch_get_status(self._h, out.ctypes.data), "hjd_batch_get_status")
        return out[:self.num_images]

    @property
    def rgb_bytes(self) -> int:
        return lib().hjd_batch_rgb_bytes(self._h)

    @property
    def scan_bytes(self) -> int:
        return lib().hjd_batch_scan_bytes(self._h)

    @property
    def pixels(self) -> int:
        return lib().hjd_batch_pixels(self._h)

    @property
    def coef_bytes(self) -> int:
        return lib().hjd_batch_coef_bytes(self._h)

    def out_size(self, i: int) -> tuple[int, int]:
        """(width, height) of image i's decoded output: the source size, or ceil(W/d) x ceil(H/d) with FLAG_SCALE_1_d;
        swapped with FLAG_EXIF_ORIENT for orientations 5-8."""
        w, h = c_uint32(), c_uint32()
        _check(lib().hjd_batch_get_out_size(self._h, i, ctypes.byref(w), ctypes.byref(h)), "hjd_batch_get_out_size")
        return w.value, h.value

    def orientation(self, i: int) -> int:
        """The EXIF orientation (1..8) image i's file states; applied to the output only with FLAG_EXIF_ORIENT."""
        o = lib().hjd_batch_get_orientation(self._h, i)
        if o < 1:
            raise HjdError(f"hjd_batch_get_orientation failed: {_err()}")
        return int(o)

    def rgb(self, i: int) -> np.ndarray:
        """RGB of image i: uint8 [out_h, out_w, 3] (out_size)."""
        if self.flags & FLAG_GRAY_OUT:
            raise HjdError("rgb(): this batch decodes one byte per pixel (FLAG_GRAY_OUT): use gray()")
        w, h = self.out_size(i)
        out = np.zeros((h, w, 3), dtype=np.uint8)
        _check(lib().hjd_batch_download_image(self._h, i, out.ctypes.data), "hjd_batch_download_image")
        return out

    def gray(self, i: int) -> np.ndarray:
        """Luma of image i (batch created with FLAG_GRAY_OUT): uint8 [out_h, out_w] (out_size), the decoded Y samples."""
        if not self.flags & FLAG_GRAY_OUT:
            raise HjdError("gray(): this batch was not created with FLAG_GRAY_OUT")
        w, h = self.out_size(i)
        out = np.zeros((h, w), dtype=np.uint8)
        _check(lib().hjd_batch_download_image(self._h, i, out.ctypes.data), "hjd_batch_download_image")
        return out

    def bmp(self, i: int) -> bytes:
        """The BMP file of image i (batch created with FLAG_BMP_OUT): what WriteBMP24 would have written."""
        n = lib().hjd_batch_bmp_bytes(self._h, i)
        out = np.zeros(max(n, 1), dtype=np.uint8)
        _check(lib().hjd_batch_download_bmp(self._h, i, out.ctypes.data), "hjd_batch_download_bmp")
        return out[:n].tobytes()

    def rgb_slab(self) -> np.ndarray:
        out = np.zeros(max(self.rgb_bytes, 1), dtype=np.uint8)
        _check(lib().hjd_batch_download_rgb(self._h, out.ctypes.data), "hjd_batch_download_rgb")
        return out[:self.rgb_bytes]

    def coefficients(self) -> np.ndarray:
        """All blocks of the batch: int16 [n_blocks, 64], zig-zag order, DC un-differenced."""
        n = self.coef_bytes // 128
        out = np.zeros((max(n, 1), 64), dtype=np.int16)
        _check(lib().hjd_batch_download_coef(self._h, out.ctypes.data), "hjd_batch_download_coef")
        return out[:n]

    def image_coefficients(self, i: int, all_coef: np.ndarray | None = None) -> np.ndarray:
        inf = self.info(i)
        c = self.coefficients() if all_coef is None else all_coef
        return c[inf.block_base:inf.block_base + inf.n_blocks]

    def image_coefficients_direct(self, i: int) -> np.ndarray:
        """Blocks of image i only (int16 [n_blocks, 64]), without downloading the whole slab."""
        inf = self.info(i)
        out = np.zeros((max(inf.n_blocks, 1), 64), dtype=np.int16)
        _check(lib().hjd_batch_download_image_coef(self._h, i, out.ctypes.data), "hjd_batch_download_image_coef")
        return out[:inf.n_blocks]

    def planes(self, i: int, slab: np.ndarray | None = None):
        """(Y, Cb, Cr) uint8 planes of image i (MCU-padded); requires FLAG_KEEP_PLANES."""
        if slab is None:
            slab = self.plane_slab()
        inf = self.info(i)
        yh = inf.mcus_y * 8 * inf.vf
        ch = inf.mcus_y * 8
        y = slab[inf.y_offset:inf.y_offset + inf.y_pitch * yh].reshape(yh, inf.y_pitch)
        if inf.ncomp == 1:
            return y, None, None
        cb = slab[inf.cb_offset:inf.cb_offset + inf.c_pitch * ch].reshape(ch, inf.c_pitch)
        cr = slab[inf.cr_offset:inf.cr_offset + inf.c_pitch * ch].reshape(ch, inf.c_pitch)
        return y, cb, cr

    def plane_slab(self) -> np.ndarray:
        n = lib().hjd_batch_plane_bytes(self._h)
        out = np.zeros(max(n, 1), dtype=np.uint8)
        _check(lib().hjd_batch_download_planes(self._h, out.ctypes.data), "hjd_batch_download_planes")
        return out[:n]

    # -- host-buffer end-to-end --------------------------------------------------------------
    def decode_host(self, arena: PinnedArena, rgb_out_ptr: int, rgb_capacity: int, chunk_images: int = 0):
        """Host buffers in, host buffers out (H2D + kernels + D2H).  Returns (offsets, status)."""
        offs = (c_uint64 * arena.n)()
        status = np.zeros(max(arena.n, 1), dtype=np.int32)
        _check(lib().hjd_batch_decode_host(self._h, arena.ptr, arena.offsets, arena.sizes, arena.n,
                                           rgb_out_ptr, rgb_capacity, offs, status.ctypes.data, chunk_images),
               "hjd_batch_decode_host")
        return np.frombuffer(offs, dtype=np.uint64).copy(), status[:arena.n]


class MultiDecoder:
    """Several GPUs in one process (hjd_multi_*): one batch handle and one host thread per device, the batch
    cut into contiguous image ranges balanced by compressed bytes; no exchange between the devices."""

    def __init__(self, devices: list[int] | None = None, flags: int = 0):
        devs = list(range(lib().hjd_device_count())) if devices is None else list(devices)
        if not devs:
            raise HjdError("no CUDA device available (this library has no CPU fallback)")
        self.devices = devs
        self._h = lib().hjd_multi_create((c_int * len(devs))(*devs), len(devs), flags)
        if not self._h:
            raise HjdError(f"hjd_multi_create failed: {_err()}")

    def close(self):
        if self._h:
            lib().hjd_multi_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def out_slab_bytes(self, arena: "PinnedArena") -> int:
        return int(lib().hjd_multi_out_slab_bytes(self._h, arena.ptr, arena.offsets, arena.sizes, arena.n))

    def decode_host(self, arena: "PinnedArena", rgb_out_ptr: int, rgb_capacity: int):
        """Host buffers in, host buffers out, all devices at once.  Returns (offsets, status)."""
        offs = (c_uint64 * arena.n)()
        status = np.zeros(max(arena.n, 1), dtype=np.int32)
        rc = lib().hjd_multi_decode_host(self._h, arena.ptr, arena.offsets, arena.sizes, arena.n, rgb_out_ptr,
                                         rgb_capacity, offs, status.ctypes.data)
        if rc != 0:
            raise HjdError(f"hjd_multi_decode_host failed ({rc}): {lib().hjd_multi_last_error(self._h).decode(errors='replace')}")
        return np.frombuffer(offs, dtype=np.uint64).copy(), status[:arena.n]


def shard_range_c(sizes: list[int], rank: int, world: int) -> tuple[int, int]:
    """The library's own sharding rule (hjd_shard_range); same result as sharding.shard_range."""
    n = len(sizes)
    lo, hi = c_int(), c_int()
    _check(lib().hjd_shard_range((c_int64 * max(n, 1))(*sizes), n, rank, world, ctypes.byref(lo), ctypes.byref(hi)), "hjd_shard_range")
    return lo.value, hi.value


def link_probe(device: int, host_in_ptr: int, h2d_bytes: int, host_out_ptr: int, d2h_bytes: int, reps: int = 3):
    """(ms_h2d, ms_d2h) per repetition of concurrent pinned copies with no kernels (hjd_link_probe)."""
    a, b = c_float(), c_float()
    _check(lib().hjd_link_probe(device, host_in_ptr, h2d_bytes, host_out_ptr, d2h_bytes, reps, ctypes.byref(a), ctypes.byref(b)),
           "hjd_link_probe")
    return a.value, b.value


def rgb_slab_bytes(arena: PinnedArena) -> int:
    return int(lib().hjd_rgb_slab_bytes(arena.ptr, arena.offsets, arena.sizes, arena.n))


def idct_matrix():
    """(M_hi, M_lo): the two integer matrices [zig-zag position k][sample 8y+x] of the tensor-core kernel, read back from the
    FP16 tile image hjd_get_idct_matrix builds (un-swizzled here): M = (M_hi * 2^11 + M_lo) * 2^-24 up to 2^-25."""
    img = np.zeros(8192, dtype=np.uint16)
    lib().hjd_get_idct_matrix(img.ctypes.data)
    h = img.view(np.float16).astype(np.float64)
    hi = np.zeros((64, 64)); lo = np.zeros((64, 64))
    for row in range(128):
        for k in range(64):
            off = (row >> 3) * 1024 + (row & 7) * 128 + (((k >> 3) ^ (row & 7)) << 4) + (k & 7) * 2
            v = h[off // 2]
            if row < 64:
                hi[k, row] = v * 8192.0
            else:
                lo[k, row - 64] = v
    return hi, lo


def idct_tables():
    c = np.zeros((8, 8), dtype=np.float32)
    cc = np.zeros((8, 8), dtype=np.float32)
    lib().hjd_get_idct_tables(c.ctypes.data, cc.ctypes.data)
    return c, cc
