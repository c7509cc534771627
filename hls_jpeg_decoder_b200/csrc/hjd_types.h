// csrc/hjd_types.h -- descriptors shared by the host boundary code and the CUDA kernels.
//
// This replaces the reference's fixed-capacity carrier structs (stJpegData / stHuffmanData /
// stComponent / stHuffmanTable, loadjpg.h:97-171): instead of one image with inline arrays,
// a batch is a set of flat HBM slabs plus one small descriptor per image.
#pragma once
#include <stdint.h>

#define HJD_LUT_BITS    10                    // first-level Huffman lookup width
#define HJD_LUT_SIZE    (1 << HJD_LUT_BITS)
#define HJD_MAX_PIXELS  (1ull << 28)          // 16384 x 16384: larger frames are rejected (a corrupt SOF must not allocate 13 GB)
#define HJD_MAX_TABLES  6                     // (DC, AC) x 3 components, de-duplicated per set

// One flattened Huffman table (built on the host from BITS/HUFFVAL, i.e. the same canonical
// codes GenHuffCodes produces, openjpg.cpp:48-66).  A first-level entry already holds what the
// symbol MEANS for the decode loop (ProcessHuffmanBlock's run/size logic, loadjpg.cpp:616-627, 768-808),
// so the kernels do no per-symbol case analysis:
//   lut[peek >> (16 - LUT_BITS)] = len | size << 5 | kadv << 9      (16 bits; 0: code longer than LUT_BITS)
//     len   code length (1..16); size = number of value bits that follow (0..15)
//     kadv  advance of the zig-zag index: DC 1; AC run+1; EOB 63 (k >= 1 in an AC position, so the block ends);
//           ZRL 16; other size-0 symbols 0 (ignored)
//   A coefficient is written at (k + kadv - 1) iff size != 0: a DC symbol with size 0 adds nothing to
//   the predictor, and the output block is zero-filled beforehand.
//   longer codes (second level): a first-level entry with len == 0 points at a sub-table:
//     sh << 5 | (offset / 2) << 8, where 6 - sh = 1..6 further bits decide;
//     lut2[offset + (the next 6 bits >> sh)] has the same layout as a first-level entry (len = full length).
//     One more shared-memory load instead of a search over the lengths: with ~12 symbols per block some
//     lane of a warp holds a long code on every other step.
//   no such code (either level): HJD_BAD_ENTRY = one bit consumed, no value, zig-zag advance 127 -- the
//     block ends there, and it ends with k >= 127, which no decodable block can (63 + 63 at most): that is
//     how the kernels recognise it, once per block instead of once per symbol (kernel 1a stops the
//     interval, kernel 1b flags the image and carries on, identically in all of its passes).
#define HJD_SYM_FIELDS(len, size, kadv) ((uint32_t)(len) | (uint32_t)(size) << 5 | (uint32_t)(kadv) << 9)
#define HJD_BAD_ENTRY   HJD_SYM_FIELDS(1, 0, 127)
#define HJD_LUT2_SIZE   512                   // canonical codes: at most 256 (one entry per long code) + 126 (sub-tables that straddle a change of length)
struct HjdHuffTable {
    uint16_t lut[HJD_LUT_SIZE];
    uint16_t lut2[HJD_LUT2_SIZE];   // sizeof == 3072, a multiple of 16 (copied to shared memory as uint4)
};

// Huffman tables of one image (or of many images that share identical DHT segments).
struct HjdTableSet {
    HjdHuffTable tab[HJD_MAX_TABLES];
    int32_t n_tabs;
    uint8_t dc_of_comp[4];   // component -> index into tab[]
    uint8_t ac_of_comp[4];
    uint8_t pad[4];
};

// Quantisation tables of one image, per component, zig-zag order (as in the file, openjpg.cpp:102-116).
// Component 1 (Cb) already carries Cr's table: the reference dequantises Cb with Cr's (loadjpg.cpp:984).
struct HjdQuantSet {
    uint16_t q[3][64];
    // the same tables packed for DP2A: word i = q[2i] | q[2i+1] << 24 (bytes 1, 2 zero), so that
    // dp2a_lo/hi(coefficient pair, word) = coef[2i]*q[2i] resp. coef[2i+1]*q[2i+1] with no unpacking
    uint32_t qp[3][32];
    // the same tables as FP16 pairs (q <= 255 is exact): word i = half(q[2i]) | half(q[2i+1]) << 16, the
    // multiplier of the tensor-core kernel's packed FP16 de-quantisation (mcu_tc.cuh)
    uint32_t qh[3][32];
};

struct HjdImageDesc {
    uint32_t width, height;
    uint32_t mcus_x, mcus_y;
    uint32_t n_mcus;
    uint32_t restart_interval;   // MCUs; 0 = whole scan is one interval
    uint32_t n_intervals;
    uint32_t interval_base;      // global index of this image's first restart interval
    uint32_t scan_len;           // entropy-coded bytes
    uint32_t table_set;          // index into the table-set pool
    uint32_t quant_set;          // index into the quant-set pool
    uint32_t y_pitch, c_pitch;   // plane pitches in bytes (MCU-padded widths)
    uint8_t  ncomp, hf, vf, blocks_per_mcu;
    uint64_t scan_off;           // byte offset of the entropy-coded segment in the file arena
    uint64_t block_base;         // first 8x8 block of this image in the coefficient slab
    uint64_t n_blocks;
    uint64_t y_off, cb_off, cr_off;   // byte offsets in the plane slab
    uint64_t rgb_off;            // byte offset in the RGB slab
    uint32_t sub_base;           // self-sync path: global index of this image's first sub-sequence
    uint32_t n_subs;             // self-sync path: sub-sequences in this image (0 = restart path)
};

// One CTA's worth of restart intervals for the entropy kernel; all share one table set.  They are
// given as segments (runs of consecutive intervals of one image): images that use the same tables are
// packed into the same CTAs even when other images lie between them in the batch, so a batch of
// small images with mixed tables (config 5: gray and colour thumbnails alternate) still fills its CTAs.
struct HjdEntropyWork {
    uint32_t first_seg;          // index into the segment array
    uint32_t n_segs;
    uint32_t n_intervals;        // sum over the segments, <= threads per CTA
    uint32_t table_set;
};
struct HjdEntropySeg {
    uint32_t first_interval;     // global interval index
    uint32_t tid0;               // thread of the CTA that takes first_interval
    uint32_t image;
    uint32_t n;                  // intervals in this segment
};

#ifndef HJD_ENT_THREADS
#define HJD_ENT_THREADS   256   // entropy kernel: one restart interval per thread
#endif
#ifndef HJD_ENT_MINBLOCKS
#define HJD_ENT_MINBLOCKS 4     // CTAs per SM the entropy kernel is compiled for (register cap)
#endif

// Marker scan of long scans: slices of HJD_SCAN_SLICE_BYTES (a multiple of the 16 KB a CTA scans per step).
#define HJD_SCAN_SLICE_MIN   (1u << 20)     // scans longer than this are sliced
#define HJD_SCAN_SLICE_BYTES (1u << 16)
struct HjdScanSlice {
    uint32_t image;
    uint32_t index;       // slice number inside the image; the slices of an image are consecutive in the list
    uint32_t n_slices;    // of that image
    uint32_t pad;
};

// ---- self-synchronising path (restart-free scans) -------------------------------------------
#define HJD_SS_SUB_BYTES   128          // sub-sequence length in (de-stuffed) bytes = 1024 bits
#define HJD_SS_MIN_BYTES   1024         // restart-free scans shorter than this stay on the 1-thread path
#define HJD_SS_SLACK       512          // zeroed bytes after every de-stuffed stream: a block that starts in the last
                                        // sub-sequence may run 63 x 26 bits past it, plus the words in flight
#define HJD_SS_THREADS     256
#ifndef HJD_SS_FIX_WARPS
#define HJD_SS_FIX_WARPS   4     // warps per CTA of the synchronisation rounds, one range of sub-sequences each
#endif
#ifndef HJD_SS_FIX_MAXR
#define HJD_SS_FIX_MAXR    256   // largest range
#endif
#define HJD_SS_FIX_OVERLAP 4     // sub-sequences before a range that its warp re-checks privately

// One per image decoded by the self-synchronising kernels; all index spaces below are global
// over the batch (sub-sequences, 16-byte de-stuffing chunks).
struct HjdSsImage {
    uint32_t img;          // image index in the batch
    uint32_t sub_base;     // first sub-sequence
    uint32_t n_subs;
    uint32_t chunk_base;   // first 16-byte chunk of the (16-byte aligned) stuffed scan
    uint32_t n_chunks;
    uint32_t lead;         // bytes between the aligned chunk origin and the first scan byte
    uint64_t dst_off;      // offset of the de-stuffed stream in the de-stuff buffer
};

// One CTA of the speculative / write kernels: segments (runs of consecutive sub-sequences of one image)
// that add up to at most HJD_SS_THREADS sub-sequences -- or of the synchronisation rounds: at most
// HJD_SS_FIX_WARPS segments, one range per warp.  All images of a CTA share one table set; images are
// grouped by table set, so a batch of small restart-free images fills its CTAs.
struct HjdSsWork {
    uint32_t first_seg;    // index into the HjdSsSeg array
    uint32_t n_segs;
    uint32_t n_subs;       // sum over the segments
    uint32_t table_set;
};
struct HjdSsSeg {
    uint32_t ss;           // index into the HjdSsImage array
    uint32_t first_sub;    // local index of the segment's first sub-sequence
    uint32_t tid0;         // thread of the CTA that takes first_sub (speculative / write kernels)
    uint32_t n;            // sub-sequences in the segment
};

// ---- multi-scan path (HJD_FLAG_MULTI_SCAN: progressive and non-interleaved files, csrc/multiscan.cu) ----------
#define HJD_MAX_SCANS      256   // scans per image; more: HJD_IMG_ERR_UNSUPPORTED (hostile files carry thousands)
#define HJD_SCAN_SEQ       0     // sequential: the block decode of kernel 1a over the scan's components
#define HJD_SCAN_DC_FIRST  1
#define HJD_SCAN_DC_REFINE 2
#define HJD_SCAN_AC_FIRST  3
#define HJD_SCAN_AC_REFINE 4

// One scan of one image.  Its MCU is the frame's MCU when it is interleaved (ncomp > 1) and one block of its
// component otherwise, on the component's own grid ceil(ceil(W h_c / h_max) / 8) x ceil(ceil(H v_c / v_max) / 8).
// Slab index of (component c, block row by, column bx): block_base + MCU * blocks_per_mcu + (luma:
// (by % vf) * hf + bx % hf, chroma: hf * vf + c - 1), the layout kernel 1a writes.
struct HjdScanDesc {
    uint32_t image;
    uint8_t  ncomp, comp[3];     // frame component indices, scan order
    uint8_t  ss, se, ah, al;
    uint8_t  kind, level, pad[2];
    uint32_t restart_interval;   // MCUs of this scan, 0 = none
    uint32_t mcus_x, mcus_y;     // this scan's MCU grid
    uint32_t n_intervals;
    uint32_t start_base;         // index of its first interval start in the batch's start table
    uint32_t scan_len;
    uint64_t scan_off;           // byte offset of the entropy-coded segment in the file arena
    uint32_t dc_tab[3], ac_tab[3];   // per scan component: index into the batch's per-scan table pool
};
// One work item = one thread of the multi-scan kernel: restart interval `interval` of scan `scan`.
struct HjdMsWork {
    uint32_t scan;
    uint32_t interval;
};

// ---- EXIF orientation (HJD_FLAG_EXIF_ORIENT, csrc/orient.cu) -----------------------------------
// One oriented image: the output kernel wrote its decoded w x h pixels at src_off (a private staging region of the
// output slab); the orientation pass writes them turned by EXIF orientation o (2..8) at dst_off, the image's place in
// the output slab.  Offsets in bytes of the output slab.
struct HjdOrientJob {
    uint64_t src_off, dst_off;
    uint32_t w, h;               // decoded size (scaled with HJD_FLAG_SCALE_*), before orientation
    uint32_t o, pad;
};
#define HJD_ORIENT_TILE 64       // the orientation pass writes output tiles of HJD_ORIENT_TILE^2 pixels, one per CTA

// Per-image status bits written by kernels (mirrors HJD_IMG_WARN_* in include/hjd.h).
#define HJD_ST_BAD_CODE     1
#define HJD_ST_COEF_RANGE   2
#define HJD_ST_OVERRUN      4
#define HJD_ST_RESTART      8
