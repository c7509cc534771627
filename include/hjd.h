/* include/hjd.h -- C ABI of the B200-native baseline-JPEG decode path.
 *
 * Drop-in boundary for the hot path of harutel/hls-jpeg-decoder (SURVEY.md 8b).  The
 * reference has plain C++ linkage and no FFI; these are the entry points a binding (cgo,
 * JNI, ctypes, ...) or the reference's own main.cpp would bind instead of its CPU decode:
 *
 *   reference interface (file:line)                           -> replacement
 *   ---------------------------------------------------------------------------------------
 *   int  ConvertJpgFile(char*, char*)        openjpg.h:23, openjpg.cpp:593  -> hjd_convert_jpg_file
 *   int  DecodeJpgFileData(buf,size,&rgb,&w,&h)  loadjpg.h:186 (declared only) -> hjd_decode_jpg_file_data
 *   void JpegGetImageSize(..., &w, &h)       loadjpg.h:183 (declared only)  -> hjd_get_image_size
 *   void WriteBMP24(name, w, h, rgb)         openjpg.cpp:504                -> hjd_write_bmp24
 *   int  JpegDecodeHW(stJpegData*, h, w, hF, vF) loadjpg.h:180, loadjpg.cpp:1134
 *        (the HLS top: parsed tables + entropy segment in, RGB out)         -> hjd_batch_* (N images per call)
 *
 * csrc/ref_shim.cpp additionally defines the reference's exact C++ names on top of this ABI
 * so that the reference's src/main.cpp links unchanged (INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only; no global mutable state besides a lazily
 * created per-thread default batch used by the single-image calls; one hjd_batch per GPU,
 * used from one host thread at a time.  All hot-path work runs in hand-written sm_100a CUDA
 * kernels; there is no CPU fallback: without a usable GPU every decode call fails with
 * HJD_ERR_CUDA and hjd_last_error() says why.
 *
 * Output contract (loadjpg.cpp:921-925): RGB24, top-down, tightly packed, stride 3*width, R first.
 * BMP contract (openjpg.cpp:504-570): 54-byte header, bottom-up rows, B,G,R, rows padded to 4 bytes.
 */
#ifndef HJD_H
#define HJD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HJD_VERSION 100

/* Return codes of the batch API (single-image reference-style calls return 1/0, see below). */
#define HJD_OK                 0
#define HJD_ERR_ARG           -1
#define HJD_ERR_CUDA          -2   /* no device / CUDA runtime failure; see hjd_last_error() */
#define HJD_ERR_NOMEM         -3
#define HJD_ERR_IO            -4
#define HJD_ERR_STATE         -5   /* call order (e.g. decode before upload) */

/* Per-image status (hjd_batch_get_status).  0 = decoded; parse errors are negative and the
 * image is skipped (its RGB slab is left zero-filled); decode warnings are positive bit flags
 * and the image is still produced (the reference itself only printf()s on such input). */
#define HJD_IMG_OK                 0
#define HJD_IMG_ERR_NOT_JPEG      -1   /* openjpg.cpp:481-486 */
#define HJD_IMG_ERR_TRUNCATED     -2
#define HJD_IMG_ERR_UNSUPPORTED   -3   /* 12-bit, 16-bit DQT, CMYK, chroma sampling != 1x1, progressive / multi-scan unless HJD_FLAG_MULTI_SCAN ... */
#define HJD_IMG_ERR_BAD_TABLE     -4   /* DHT over-subscribed / missing table */
#define HJD_IMG_WARN_BAD_CODE      1   /* undecodable Huffman code; rest of that restart interval zero-filled */
#define HJD_IMG_WARN_COEF_RANGE    2   /* run past coefficient 63 (loadjpg.cpp:780-783); multi-scan: run past Se, refinement size != 1 */
#define HJD_IMG_WARN_OVERRUN       4   /* entropy data ended before the interval did */
#define HJD_IMG_WARN_RESTART       8   /* RSTn count differs from ceil(MCUs/Ri)-1 */

/* hjd_batch_create flags */
#define HJD_FLAG_KEEP_PLANES   1u   /* unfused kernels 2 and 3 with the Y/Cb/Cr planes in HBM (parity tap, hjd_batch_download_planes) */
#define HJD_FLAG_HOST_SCAN     2u   /* find RSTn markers on the host instead of the GPU pre-pass */
#define HJD_FLAG_FUSED_MCU    16u   /* (default behaviour) kernels 2+3 fused per MCU: one thread decodes a whole MCU to RGB */
#define HJD_FLAG_BMP_OUT      32u   /* the output slab holds, per image, the BMP FILE WriteBMP24 would write (openjpg.cpp:504-570:
                                       54-byte header, bottom-up B G R rows padded to 4 bytes) instead of top-down RGB24: written by
                                       the colour kernel's epilogue, so a file writer only has to fwrite it.  The file of image i
                                       is hjd_batch_bmp_bytes(i) bytes from rgb_offset + 10 of the slab (pixel array 64-byte aligned). */
#define HJD_FLAG_TENSOR_CORE_IDCT 128u /* always the fused kernel with the IDCT's fast tier as tcgen05.mma on the tensor cores (csrc/mcu_tc.cuh) */
#define HJD_FLAG_CUDA_CORE_IDCT   64u  /* always the fused kernel with the fast tier as FP32 FMA chains on the CUDA cores (csrc/kernels.cu);
                                          default: chosen per chunk -- tensor cores for large colour images, CUDA cores for batches of small ones (same bytes out) */
#define HJD_FLAG_NO_SELFSYNC   8u   /* restart-free scans: one thread per scan (kernel 1a) instead of kernel 1b */
#define HJD_FLAG_MULTI_SCAN  256u   /* also decode progressive (SOF2, 8-bit Huffman) files and sequential files whose components come
                                       in separate scans (csrc/multiscan.cu; one thread per restart interval of each scan).  Such a
                                       file decodes exactly like its baseline twin, the single interleaved scan with the same quantised
                                       coefficients: same coefficients, planes, RGB and BMP bytes.  Blocks no scan codes stay 0; a file
                                       that ends early is decoded from the scans it has.  hjd_image_info of such an image:
                                       scan_bytes = the sum over its scans, restart_interval = the DRI of its first scan, n_intervals =
                                       its work items (restart intervals summed over the scans).  Single-scan baseline files take the
                                       default path unchanged.  At most HJD_MAX_SCANS_PER_IMAGE scans per file. */
#define HJD_MAX_SCANS_PER_IMAGE 256
/* Reduced-size decode in the DCT domain (a 2-bit field; 0 = full size).  With d = 2, 4 or 8 and N = 8/d samples per
 * block side, a W x H image decodes to ceil(W/d) x ceil(H/d) RGB24 in the usual layout (top-down, stride 3 * out_w,
 * R first, each image 256-byte aligned in the slab; hjd_batch_get_out_size).  Each block is de-quantised as the full
 * decode does it (Cb with Cr's table) and its top-left N x N natural-order coefficients go through the reference's
 * direct-form IDCT with N in place of 8: float sum over u < N (outer), v < N (inner) of
 * cc[u][v] * arr[u][v] * cosN[x][u] * cosN[y][v], cosN[p][k] = cosf(((2p+1) * k * 3.14f) / (2N)), then (int16) of
 * (int) of 0.25 * sum, + 128, clamp.  Per MCU the luma tile is (N hf) x (N vf) and the chroma tile N x N, upsampled by
 * the reference's replication rule with 8 replaced by N; the colour conversion is the reference's.  N = 8 would be the
 * full decode.  Every Huffman symbol of a sequential scan is still decoded (csrc/scaled.cu).
 * With HJD_FLAG_MULTI_SCAN, scans are decoded as without a scale flag, except at 1/8, where an image's AC scans
 * (Ss > 0) are not read at all: its coefficient slab holds only what its DC scans code, hjd_batch_num_scans and
 * n_intervals count its DC scans only, and damage inside an AC scan is not reported.
 * Not combinable (hjd_batch_create fails with HJD_ERR_ARG): HJD_FLAG_KEEP_PLANES (no scaled planes exist),
 * HJD_FLAG_BMP_OUT, HJD_FLAG_TENSOR_CORE_IDCT and HJD_FLAG_CUDA_CORE_IDCT (they select full-size kernels). */
#define HJD_FLAG_SCALE_1_2   (1u << 9)
#define HJD_FLAG_SCALE_1_4   (2u << 9)
#define HJD_FLAG_SCALE_1_8   (3u << 9)
#define HJD_FLAG_SCALE_MASK  (3u << 9)
/* Single-channel luma output (the grayscale read mode of libjpeg's JCS_GRAYSCALE, nvJPEG's NVJPEG_OUTPUT_Y): a W x H
 * image decodes to W x H bytes (with HJD_FLAG_SCALE_1_d: ceil(W/d) x ceil(H/d)), top-down rows, stride = output width,
 * each image 256-byte aligned in the slab at rgb_offset.  Pixel (x, y) is the Y sample (x, y) the full decode computes
 * before colour conversion: the reference's IDCT of the luma blocks with the luma table, +128, clamp -- exactly the Y
 * plane of HJD_FLAG_KEEP_PLANES, cropped from the MCU-padded plane to W x H.  A one-component file outputs its only
 * component (= each channel of its RGB decode).  With a scale flag: the luma samples of the scaled decode.  Not a
 * weighted sum of R, G and B.
 * With HJD_FLAG_MULTI_SCAN, a scan none of whose components is the frame's first is not read: it gets no work items, is
 * not counted by hjd_batch_num_scans or n_intervals, damage inside it is not reported, and the coefficients only it
 * codes stay 0.  Interleaved scans (sequential ones, a DC scan of Y, Cb and Cr) are read whole.  With
 * HJD_FLAG_SCALE_1_8 both rules apply.
 * Combines with HJD_FLAG_MULTI_SCAN, HJD_FLAG_SCALE_*, HJD_FLAG_HOST_SCAN and HJD_FLAG_NO_SELFSYNC.  Not combinable
 * (hjd_batch_create fails with HJD_ERR_ARG): HJD_FLAG_BMP_OUT (an 8-bit palettised BMP is not WriteBMP24's format),
 * HJD_FLAG_KEEP_PLANES (the planes already hold Y), HJD_FLAG_TENSOR_CORE_IDCT and HJD_FLAG_CUDA_CORE_IDCT (they select
 * RGB kernels). */
#define HJD_FLAG_GRAY_OUT    (1u << 11)
/* Apply each image's EXIF orientation to its decoded output (torchvision's apply_exif_orientation, PIL.ImageOps.
 * exif_transpose).  The orientation o is read from the first APP1 segment before the first SOS whose payload starts
 * with "Exif\0\0": the TIFF header after those 6 bytes ("II*\0" or "MM\0*", then the 32-bit offset of IFD0, relative
 * to the header), and in IFD0 (16-bit entry count, 12-byte entries tag, type, count, value) the entry with tag 0x0112,
 * type SHORT (3) and count 1: the first two bytes of its value field, in the file's byte order.  In every other case
 * o = 1: no Exif APP1 before the first SOS; an offset, count or entry reaching past the segment; another type or
 * count; a value outside 1..8; the tag only in another IFD (ExifIFD, IFD1).  A malformed tag is never an error.
 * With the decoded output W' x H' (the source size, or ceil(W/d) x ceil(H/d) with HJD_FLAG_SCALE_1_d) and bpp bytes
 * per pixel (3, or 1 with HJD_FLAG_GRAY_OUT), output pixel out(x, y) is, by o (EXIF 2.3 / TIFF 6.0):
 *   1 as stored             W' x H'  in(x, y)              5 transpose          H' x W'  in(y, x)
 *   2 mirror horizontally   W' x H'  in(W'-1-x, y)         6 rotate 90 cw       H' x W'  in(y, H'-1-x)
 *   3 rotate 180            W' x H'  in(W'-1-x, H'-1-y)    7 transverse         H' x W'  in(W'-1-y, H'-1-x)
 *   4 mirror vertically     W' x H'  in(x, H'-1-y)         8 rotate 90 ccw      H' x W'  in(W'-1-y, x)
 * Each image keeps its region of the slab (same rgb_offset, 256-byte alignment, hjd_batch_rgb_bytes and
 * hjd_out_slab_bytes); its rows are top-down with stride out_w * bpp, and hjd_batch_get_out_size returns the oriented
 * size.  hjd_image_info and hjd_batch_pixels keep describing the source.  Without the flag nothing changes, also for
 * files that carry a tag.  Combines with every flag but HJD_FLAG_BMP_OUT (hjd_batch_create fails with HJD_ERR_ARG);
 * with HJD_FLAG_KEEP_PLANES the planes stay as stored and only the RGB slab is oriented.  hjd_batch_decode_host and
 * the hjd_multi_* calls follow the handle's flags.  The single-image calls and the file converter do not orient. */
#define HJD_FLAG_EXIF_ORIENT (1u << 12)

typedef struct hjd_batch hjd_batch;

typedef struct hjd_image_info {
    uint32_t width, height;
    uint8_t  ncomp;            /* 1 or 3 */
    uint8_t  hf, vf;           /* luma sampling factors (1 or 2); chroma is 1x1 */
    uint8_t  blocks_per_mcu;
    uint32_t mcus_x, mcus_y;
    uint32_t restart_interval; /* MCUs, 0 = none */
    uint32_t n_intervals;
    uint32_t scan_bytes;       /* entropy-coded segment length */
    uint64_t block_base;       /* first block of this image in the coefficient buffer */
    uint64_t n_blocks;
    uint64_t rgb_offset;       /* byte offset of this image in the RGB slab */
    uint64_t y_offset, cb_offset, cr_offset;   /* byte offsets in the plane slab */
    uint32_t y_pitch, c_pitch;
    int32_t  status;
} hjd_image_info;

/* Stage timings of the last hjd_batch_decode (CUDA events on the batch stream), milliseconds. */
typedef struct hjd_timings {
    float scan_ms;      /* kernel 0: RSTn marker scan -> interval table */
    float entropy_ms;   /* kernel 1: Huffman decode -> int16 coefficients (+ self-sync passes) */
    float idct_ms;      /* kernel 2 (or fused 2+3) */
    float color_ms;     /* kernel 3 (0 when fused) */
    float total_ms;
    int   launches;     /* kernels launched by the last decode */
} hjd_timings;

/* ---- library ---------------------------------------------------------------------------- */
int         hjd_version(void);
const char* hjd_last_error(void);          /* thread-local, never NULL */
int         hjd_device_count(void);        /* 0 when no CUDA device is usable */

/* ---- reference-shaped single-image entry points (return 1 = success, 0 = failure) -------- */
/* openjpg.cpp:593 ConvertJpgFile: load .jpg, decode on the GPU, write 24-bit .bmp. */
int  hjd_convert_jpg_file(const char* jpg_in, const char* bmp_out);
/* loadjpg.h:186 DecodeJpgFileData: *rgb is allocated by the library (release with hjd_free). */
int  hjd_decode_jpg_file_data(const uint8_t* buf, int size, uint8_t** rgb, unsigned* width, unsigned* height);
void hjd_free(void* p);
/* Same, with the result allocated by the caller's allocator (the C++ shim passes operator new[], so that the
 * reference's "delete[] rgbpix" contract holds without a second copy). */
int  hjd_decode_jpg_file_data_alloc(const uint8_t* buf, int size, void* (*alloc)(size_t), uint8_t** rgb,
                                    unsigned* width, unsigned* height);
/* Device used by the reference-shaped single-image calls (a lazily created per-thread batch); default 0. */
int  hjd_set_default_device(int device);
/* loadjpg.h:183 JpegGetImageSize, from the file bytes (header parse only, no GPU). */
int  hjd_get_image_size(const uint8_t* buf, int size, unsigned* width, unsigned* height);
/* Header parse only (no GPU): the per-image status a batch would report for this file (HJD_IMG_OK or a
 * negative HJD_IMG_ERR_*) and, when it is decodable, its geometry (offsets in *out stay 0).
 * Not decodable: lossless / arithmetic (SOF3, SOF5..SOF15), 12-bit samples (SOF1 with P != 8), 16-bit DQT,
 * 4 components, chroma sampling other than 1x1, luma factors other than 1 or 2; and, unless HJD_FLAG_MULTI_SCAN,
 * progressive files (SOF2) and NON-INTERLEAVED baseline files (one scan per component): the reference's decode
 * loop is one interleaved scan of all three components (loadjpg.cpp:945-997), so without the flag such files get
 * HJD_IMG_ERR_UNSUPPORTED. */
int  hjd_probe_jpeg(const uint8_t* buf, int64_t size, hjd_image_info* out);
/* The same for a batch created with `flags` (flags 0: identical to hjd_probe_jpeg).  No GPU. */
int  hjd_probe_jpeg_flags(const uint8_t* buf, int64_t size, unsigned flags, hjd_image_info* out);
/* The scans of a file as a batch with HJD_FLAG_MULTI_SCAN decodes them (no GPU): up to `max` into out[], in file
 * order.  comp[] are frame component indices; level: the scan's dependency level (scans of one level write
 * disjoint coefficients and are decoded by one launch); restart_interval: the DRI in effect at that scan; bytes:
 * its entropy-coded segment.  Returns the number of scans (a single-scan baseline file: 1), or the negative
 * per-image status of a file that is not decodable. */
typedef struct hjd_scan_info {
    uint8_t  ncomp, comp[3];
    uint8_t  ss, se, ah, al;
    uint8_t  level, pad[3];
    uint32_t restart_interval, bytes;
} hjd_scan_info;
int  hjd_probe_jpeg_scans(const uint8_t* buf, int64_t size, hjd_scan_info* out, int max);
/* The EXIF orientation (1..8) the file states, by the rule of HJD_FLAG_EXIF_ORIENT (header parse only, no GPU);
 * HJD_IMG_ERR_NOT_JPEG when the buffer does not start with SOI. */
int  hjd_probe_jpeg_orientation(const uint8_t* buf, int64_t size);
/* openjpg.cpp:504 WriteBMP24. */
int  hjd_write_bmp24(const char* path, unsigned width, unsigned height, const uint8_t* rgb);
/* Same bytes as hjd_write_bmp24 into memory; returns the BMP size (call with out = NULL to size it). */
size_t hjd_encode_bmp24(unsigned width, unsigned height, const uint8_t* rgb, uint8_t* out);

/* ConvertJpgFile at batch scale, as a pipeline (openjpg.cpp:593-684 per file): `threads` readers fill a pinned
 * arena; per device up to three workers decode one chunk of `chunk_images` images at a time with
 * HJD_FLAG_BMP_OUT (the GPU writes the BMP file layout); `threads` writers fwrite every file as soon as its
 * chunk has landed in pinned memory, while later chunks are being copied and decoded (0 = all cores / 32
 * images).  ok[i] = 1 / 0 per file (may be NULL).  Returns the number of files converted. */
int  hjd_convert_jpg_files(const char* const* jpg_in, const char* const* bmp_out, int n, int device,
                           int threads, int* ok);
int  hjd_convert_jpg_files_multi(const char* const* jpg_in, const char* const* bmp_out, int n,
                                 const int* devices, int n_devices, int threads, int chunk_images, int* ok);

/* ---- batch API: the JpegDecodeHW replacement, N independent images per call -------------- */
hjd_batch* hjd_batch_create(int device, unsigned flags);
void       hjd_batch_destroy(hjd_batch* b);
/* Use an existing CUDA stream (cudaStream_t passed as void*) instead of the batch's own. */
int  hjd_batch_set_stream(hjd_batch* b, void* cuda_stream);

/* Parse headers, build Huffman/quant tables and descriptors, copy the files to HBM.
 * bufs[i]/sizes[i]: whole .jpg files in host memory (pinned memory makes the copy asynchronous).
 * Limits per batch (HJD_ERR_ARG, naming the limit, before anything is allocated or copied): fewer than 2^32 blocks;
 * restart-free scans fitting in fewer than 2^32 16-byte chunks (about 64 GiB); with HJD_FLAG_MULTI_SCAN, fewer than
 * 2^31 multi-scan work items (restart intervals of all scans).  DESIGN.md §3 "Index limits". */
int  hjd_batch_upload(hjd_batch* b, const uint8_t* const* bufs, const int64_t* sizes, int n);
/* Same, for files packed in one host arena: file i = arena[offsets[i] .. offsets[i]+sizes[i]).
 * One host->device copy of [offsets[0], offsets[n-1]+sizes[n-1]). */
int  hjd_batch_upload_arena(hjd_batch* b, const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n);

/* Launch the decode of everything uploaded (asynchronous on the batch stream):
 * marker scan -> entropy decode -> dequant/IDCT -> upsample/colour.  Results stay in HBM. */
int  hjd_batch_decode(hjd_batch* b);
int  hjd_batch_sync(hjd_batch* b);
/* hjd_batch_decode_host splits large batches into up to 8 chunks on 3 streams so that the H2D copy,
 * the kernels and the D2H copy of different chunks overlap (default, on = 1).  HBM-resident decodes
 * (hjd_batch_upload* + hjd_batch_decode) run on one stream, in order: measured on B200, overlapping
 * their kernels gains nothing (all are issue-bound) and per-stage timings need the serial order.
 * on = 0: never chunk; on > 1: chunk both paths with this target number of 8x8 blocks per chunk
 * (testing / tuning).  Takes effect at the next upload. */
int  hjd_batch_set_overlap(hjd_batch* b, int on);

/* Synchronisation rounds the self-synchronising kernel (restart-free scans) needed in the last decode. */
int  hjd_batch_selfsync_rounds(hjd_batch* b);                        /* syncs */
/* Sub-sequences per warp in those rounds: 0 = pick by batch size (default), else a multiple of 32 up
 * to 256 (testing / tuning; results do not depend on it).  Takes effect at the next upload. */
int  hjd_batch_set_selfsync_range(hjd_batch* b, int range);
/* Which fused kernel(s) the chunks of the last decode went through: bit 0 = tensor cores (csrc/mcu_tc.cuh), bit 1 = CUDA
 * cores, bit 2 = the scaled kernel (HJD_FLAG_SCALE_*, csrc/scaled.cu), bit 3 = a luma-only kernel (HJD_FLAG_GRAY_OUT;
 * with a scale flag set together with bit 2); 0 = none (nothing decoded yet, or HJD_FLAG_KEEP_PLANES). */
int  hjd_batch_idct_variant(const hjd_batch* b);
int  hjd_batch_num_images(const hjd_batch* b);
/* Scans image i of the last upload is decoded from (1: single-scan baseline; 0: not decodable).  HJD_FLAG_SCALE_1_8
 * with HJD_FLAG_MULTI_SCAN: its DC scans only; HJD_FLAG_GRAY_OUT with HJD_FLAG_MULTI_SCAN: the scans that contain luma. */
int  hjd_batch_num_scans(const hjd_batch* b, int i);
/* hjd_image_info describes the source image (width, height: its frame). */
int  hjd_batch_get_info(const hjd_batch* b, int i, hjd_image_info* out);
/* Dimensions of image i's decoded output: width x height, or ceil(width/d) x ceil(height/d) with HJD_FLAG_SCALE_1_d
 * (the same with HJD_FLAG_GRAY_OUT); with HJD_FLAG_EXIF_ORIENT and orientation 5..8, width and height swapped. */
int  hjd_batch_get_out_size(const hjd_batch* b, int i, uint32_t* w, uint32_t* h);
/* The EXIF orientation (1..8) image i's file states, with or without HJD_FLAG_EXIF_ORIENT (which decides only whether
 * it is applied); negative (HJD_ERR_ARG) for a bad index. */
int  hjd_batch_get_orientation(const hjd_batch* b, int i);
int  hjd_batch_get_status(hjd_batch* b, int32_t* status /* n */);   /* syncs */
int  hjd_batch_get_timings(hjd_batch* b, hjd_timings* out);          /* syncs */
/* CUDA-event stopwatch on the batch stream: record event `slot` (0..HJD_MARK_SLOTS-1); milliseconds
 * between two recorded slots (waits for slot_b).  This is how bench.py times K steps, and each of
 * them, on the launching stream. */
#define HJD_MARK_SLOTS 130
int   hjd_batch_mark(hjd_batch* b, int slot);
float hjd_batch_elapsed_ms(hjd_batch* b, int slot_a, int slot_b);
uint64_t hjd_batch_rgb_bytes(const hjd_batch* b);     /* size of the RGB slab (the output slab: 1 byte per pixel with HJD_FLAG_GRAY_OUT) */
uint64_t hjd_batch_coef_bytes(const hjd_batch* b);
uint64_t hjd_batch_plane_bytes(const hjd_batch* b);
uint64_t hjd_batch_scan_bytes(const hjd_batch* b);    /* sum of entropy-coded bytes */
uint64_t hjd_batch_pixels(const hjd_batch* b);        /* sum of width*height (source pixels, also when scaled) */

/* Device pointers of the result slabs (valid until the next upload / destroy). */
void* hjd_batch_device_rgb(hjd_batch* b);
void* hjd_batch_device_coef(hjd_batch* b);
void* hjd_batch_device_planes(hjd_batch* b);

/* Device -> host copies (synchronous with respect to the batch stream). */
int  hjd_batch_download_rgb(hjd_batch* b, uint8_t* dst /* hjd_batch_rgb_bytes */);
int  hjd_batch_download_image(hjd_batch* b, int i, uint8_t* dst /* out_w*out_h*3 (HJD_FLAG_GRAY_OUT: out_w*out_h),
                                                                    hjd_batch_get_out_size */);
int  hjd_batch_download_coef(hjd_batch* b, int16_t* dst /* hjd_batch_coef_bytes */);
uint64_t hjd_batch_bmp_bytes(const hjd_batch* b, int i);            /* HJD_FLAG_BMP_OUT: size of image i's BMP file (0: none) */
int  hjd_batch_download_bmp(hjd_batch* b, int i, uint8_t* dst /* hjd_batch_bmp_bytes(i) */);
int  hjd_batch_download_image_coef(hjd_batch* b, int i, int16_t* dst /* n_blocks*64 */);   /* one image of the slab */
int  hjd_batch_download_planes(hjd_batch* b, uint8_t* dst /* hjd_batch_plane_bytes */);

/* End to end with host buffers: upload, decode and download in overlapped chunks
 * (copy engines and SMs busy at the same time).  rgb_out receives image i at
 * rgb_offsets_out[i] (tightly packed, 256-byte aligned starts); capacity in bytes. */
int  hjd_batch_decode_host(hjd_batch* b, const uint8_t* arena, const int64_t* offsets, const int64_t* sizes,
                           int n, uint8_t* rgb_out, uint64_t rgb_capacity, uint64_t* rgb_offsets_out,
                           int32_t* status_out, int chunk_images);
/* Bytes hjd_batch_decode_host needs in rgb_out for these files (header parse only); hjd_out_slab_bytes: the
 * same for a batch created with `flags` (HJD_FLAG_BMP_OUT changes the layout, HJD_FLAG_SCALE_* the output size,
 * HJD_FLAG_GRAY_OUT the bytes per pixel: align_up(out_w * out_h, 256) per image).  The hjd_multi_* calls follow the
 * flags of their handle in the same way. */
uint64_t hjd_rgb_slab_bytes(const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n);
uint64_t hjd_out_slab_bytes(const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n, unsigned flags);

/* ---- several GPUs in one process (SURVEY.md 8e) -------------------------------------------
 * Images are independent and there is no exchange step: a batch is cut into one contiguous image range per
 * device, balanced by compressed bytes (hjd_shard_range), and every device decodes its range with its own
 * hjd_batch, driven by its own host thread.  rgb_out receives the shards back to back: image i is at
 * rgb_offsets_out[i], exactly the bytes a single-device decode produces for it. */
typedef struct hjd_multi hjd_multi;
int        hjd_shard_range(const int64_t* sizes, int n, int rank, int world, int* lo, int* hi);
hjd_multi* hjd_multi_create(const int* devices /* NULL: 0..n-1 */, int n_devices, unsigned flags);
void       hjd_multi_destroy(hjd_multi* m);
int        hjd_multi_num_devices(const hjd_multi* m);
hjd_batch* hjd_multi_batch(hjd_multi* m, int k);      /* the k-th device's batch handle (resident use, timings) */
const char* hjd_multi_last_error(const hjd_multi* m);
uint64_t   hjd_multi_out_slab_bytes(const hjd_multi* m, const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n);
int        hjd_multi_decode_host(hjd_multi* m, const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n,
                                 uint8_t* rgb_out, uint64_t rgb_capacity, uint64_t* rgb_offsets_out, int32_t* status_out);

/* Pinned host memory helpers (cudaHostAlloc, portable: pinned for every device of the process / cudaFreeHost) for callers without a CUDA binding. */
void* hjd_host_alloc(size_t bytes);
void  hjd_host_free(void* p);
/* Same, with the pages taken from the NUMA node next to `device` where the platform exposes one
 * (hjd_device_numa_node: -1 otherwise): the D2H copy of the decoded batch is the end-to-end bottleneck. */
void* hjd_host_alloc_near(int device, size_t bytes);
int   hjd_device_numa_node(int device);
/* Raw host-link probe, no kernels: reps x (h2d_bytes up || d2h_bytes down, pinned buffers, two streams);
 * milliseconds per repetition and direction.  The ceiling hjd_batch_decode_host works against. */
int   hjd_link_probe(int device, const void* host_in, size_t h2d_bytes, void* host_out, size_t d2h_bytes,
                     int reps, float* ms_h2d, float* ms_d2h);

/* Testing aid: build the kernels' two-level lookup table from BITS / HUFFVAL (as in a DHT segment) and look
 * up the next 16 bits of a stream: returns len | size << 5 | zig-zag advance << 9 (0xFE01: no such code;
 * 0xFFFFFFFF: the table is over-subscribed).  tests/ compare it with the canonical code walk. */
uint32_t hjd_huff_lookup_probe(const uint8_t bits[16], const uint8_t* vals, int nvals, int is_ac, uint32_t peek16);

/* The float constants the kernels use (computed on the host with the libm expressions of
 * loadjpg.cpp:96-102,120): cos_tab[p*8+k] = cosf(((2p+1)*k*3.14f)/16), cc[u*8+v] = C(u)*C(v). */
void hjd_get_idct_tables(float cos_tab[64], float cc[64]);
/* The IDCT matrix of the tensor-core kernel as the 16 KB FP16 tile image it multiplies by (csrc/mcu_tc.cuh): with
 * M[k][8y+x] = 0.25 * cc * cos[x][u] * cos[y][v] for zig-zag position k = (u, v) (the real-number product of the constants
 * above), row n of 128 holds M_hi * 2^-13 (n = 8y+x) or M_lo (n = 64 + 8y+x), integers with M = (M_hi * 2^11 + M_lo) * 2^-24
 * up to 2^-25; 64 FP16 per row in zig-zag order, 16-byte chunk j of row n stored at chunk j ^ (n & 7), rows in 1024-byte
 * groups of eight (the K-major, 128-byte-swizzled operand layout of tcgen05.mma).  Host computation, no GPU needed. */
void hjd_get_idct_matrix(uint16_t img[8192]);

#ifdef __cplusplus
}
#endif
#endif /* HJD_H */
