// csrc/batch_plan.h -- host planning of one batch upload: header parse, table and quantisation sets, slab layout,
// chunk plan, index-limit guards and the kernels' work lists.
//
// No CUDA here: the plan is plain host data that hjd_api.cu sizes the device slabs from and copies to the GPU.  A batch
// the plan refuses has therefore taken no device memory, and the planner runs (and is tested) on machines without a GPU.
#pragma once
#include <stdint.h>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>
#include "hjd_types.h"
#include "jpeg_parse.h"
#include "../../include/hjd.h"

static inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// log2 of the scale denominator of HJD_FLAG_SCALE_* (0: full size), and the output size of a W x H image under it:
// ceil(W / d) x ceil(H / d), libjpeg's jdiv_round_up.
static inline int scale_shift(unsigned flags) { return (int)((flags & HJD_FLAG_SCALE_MASK) >> 9); }
static inline uint32_t scaled_dim(unsigned flags, uint32_t v)
{
    const int s = scale_shift(flags);
    return (uint32_t)(((uint64_t)v + (1u << s) - 1) >> s);
}

// Bytes of one image's region in the output slab: tightly packed RGB24 (of the scaled size with HJD_FLAG_SCALE_*), one
// byte per pixel (HJD_FLAG_GRAY_OUT), or (HJD_FLAG_BMP_OUT) the BMP file WriteBMP24 would write, placed so that its
// pixel array starts 64 bytes into the region (the 54-byte header at +10): rows padded to a multiple of 4 bytes,
// openjpg.cpp:534-535.
static inline uint64_t image_out_bytes(unsigned flags, uint32_t w, uint32_t h)
{
    if (flags & HJD_FLAG_BMP_OUT) return 64 + (uint64_t)((w * 3 + 3) & ~3u) * h;
    return (uint64_t)scaled_dim(flags, w) * scaled_dim(flags, h) * ((flags & HJD_FLAG_GRAY_OUT) ? 1 : 3);
}

// Whether a multi-scan batch created with `flags` reads scan `s`: at 1/8 a block is its DC coefficient alone, so the AC
// scans (Ss > 0) are not; a luma-only decode (HJD_FLAG_GRAY_OUT) does not read the scans without the frame's first
// component.
static inline bool scan_is_read(unsigned flags, const HjdScanParsed& s)
{
    if (scale_shift(flags) == 3 && s.ss > 0) return false;
    if (flags & HJD_FLAG_GRAY_OUT) {
        for (int k = 0; k < s.ncomp; k++)
            if (s.comp[k] == 0) return true;
        return false;
    }
    return true;
}

// Work items of one scan: the restart intervals its DRI implies (want_all) or, by default, no more than the file holds.
uint32_t ms_scan_items(const HjdParsed& frame, const HjdScanParsed& p, uint32_t* mcus_x, uint32_t* mcus_y,
                       bool want_all = false);

// MCU geometry of a frame (loadjpg.cpp:1170-1174) and the restart intervals of its one interleaved scan.
struct FrameGeometry { uint32_t blocks_per_mcu, mcus_x, mcus_y, n_mcus, n_intervals; };
FrameGeometry frame_geometry(uint32_t width, uint32_t height, int ncomp, int hf, int vf, uint32_t restart_interval);

// Size of an image's decoded output (hjd_batch_get_out_size): the scaled size of its w x h frame, with width and height
// swapped when HJD_FLAG_EXIF_ORIENT applies an orientation 5..8 (o: what its file states).
static inline void out_size(unsigned flags, uint32_t w, uint32_t h, int o, uint32_t* out_w, uint32_t* out_h)
{
    const bool swap = (flags & HJD_FLAG_EXIF_ORIENT) && o >= 5;
    *out_w = scaled_dim(flags, swap ? h : w);
    *out_h = scaled_dim(flags, swap ? w : h);
}

// Output tiles of the orientation pass (csrc/orient.cu) of an out_w x out_h image.
static inline uint32_t orient_tiles(uint32_t out_w, uint32_t out_h)
{
    return ((out_w + HJD_ORIENT_TILE - 1) / HJD_ORIENT_TILE) * ((out_h + HJD_ORIENT_TILE - 1) / HJD_ORIENT_TILE);
}

// Luma blocks that hold at least one pixel of a W x H image: ceil(W/8) x ceil(H/8) (the full-size luma kernel's threads).
static inline uint64_t luma_blocks(uint32_t w, uint32_t h) { return (uint64_t)((w + 7) / 8) * ((h + 7) / 8); }

struct FileRef { const uint8_t* ptr; int64_t size; uint64_t dev_off; };

// A contiguous range of images that is uploaded / decoded / downloaded as one unit on one stream.
// Chunks of one batch use disjoint regions of the same slabs, so they can be in flight together:
// copy engines and SMs overlap, and the memory-bound colour kernel of one chunk shares the SMs with
// the issue-bound entropy / IDCT kernels of another.
struct Chunk {
    int img0 = 0, img1 = 0;
    uint32_t work0 = 0, work1 = 0;
    uint32_t slice0 = 0, slice1 = 0;          // marker-scan slices of this chunk's long scans
    uint64_t arena_lo = 0, arena_hi = 0;      // device arena byte range holding these files
    uint64_t rgb_lo = 0, rgb_hi = 0;
    uint32_t max_blocks = 0, max_w = 0, max_h = 0, max_mcus = 0;
    uint32_t max_luma = 0;                    // most luma blocks inside W x H of one image (HJD_FLAG_GRAY_OUT kernel grid)
    uint64_t blocks = 0;
    // kernel 1b (restart-free images of this chunk): ranges in the batch-wide index spaces, each with a gap of
    // one entry behind it so that the chunks' prefix sums (which append a sentinel) can run side by side
    uint32_t ss0 = 0, ss1 = 0;                // entries of BatchPlan::ss
    uint32_t sub0 = 0, n_subs = 0;            // sub-sequences
    uint32_t ck0 = 0, n_ck = 0;               // 16-byte de-stuffing chunks
    uint32_t sw0 = 0, sw1 = 0, sf0 = 0, sf1 = 0;   // work items: speculative / write kernels, synchronisation kernel
    uint32_t ss_range = 0;                    // sub-sequences per warp in the synchronisation kernel
    // multi-scan images of this chunk: their slab blocks (zeroed before the first level), their work items per level
    std::vector<std::pair<uint64_t, uint64_t>> ms_zero;     // (first block, blocks)
    std::vector<std::pair<uint32_t, uint32_t>> ms_levels;   // work item range of each level present, in level order
    uint32_t oj0 = 0, oj1 = 0;                // HJD_FLAG_EXIF_ORIENT: this chunk's entries of BatchPlan::orient_jobs
};

// What the planner is asked for.
struct PlanConfig {
    unsigned flags = 0;            // HJD_FLAG_* of the batch
    int overlap = 1;               // hjd_batch_set_overlap: 0 one chunk, 1 default chunking, > 1 target blocks per chunk
    int chunk_images = 0;          // > 0: images per chunk (hjd_batch_decode_host)
    uint32_t ss_range_req = 0;     // hjd_batch_set_selfsync_range, 0 = automatic
    int sm_count = 148;            // multiprocessors of the device (work-list balancing)
    bool chunked = false;          // plan several chunks (else one)
};

// Everything one upload computes on the host.  Per image unless noted; batch-wide index spaces as in DESIGN §3.
struct BatchPlan {
    std::vector<HjdImageDesc> imgs;
    std::vector<int32_t> parse_status;
    std::vector<HjdTableSet> tsets;
    std::vector<HjdQuantSet> qsets;
    std::unordered_multimap<uint64_t, uint32_t> tset_of, qset_of;   // content hash -> candidate sets (verified byte for byte)
    std::vector<HjdRawTables> tset_raw, qset_raw;                    // what each set was built from
    std::vector<HjdEntropyWork> work;
    std::vector<HjdEntropySeg> segs;
    std::vector<HjdScanSlice> slices;    // marker-scan slices of long restart-marker scans
    std::vector<uint32_t> mcu_cta;       // exclusive prefix of the per-image MCU counts (n + 1), for the flat grid of the per-MCU kernel
    std::vector<uint32_t> luma_cta;      // HJD_FLAG_GRAY_OUT: the same for the luma blocks inside W x H (luma_blocks), per-block kernel
    std::vector<uint32_t> host_istart;   // HJD_FLAG_HOST_SCAN only
    std::vector<uint8_t> host_restart_warn;     // HJD_FLAG_HOST_SCAN only (and multi-scan images)
    // kernel 1b
    std::vector<HjdSsImage> ss;          // images on the self-synchronising path
    std::vector<HjdSsWork> sswork;       // one entry per CTA: speculative / write kernels, then synchronisation rounds
    std::vector<HjdSsSeg> sssegs;        // their segments
    uint32_t ss_subs = 0, ss_chunks = 0; // batch-wide totals, including one gap per chunk
    uint32_t ss_tmp_stride = 0;          // words of prefix-sum scratch per chunk
    uint64_t ss_dst_bytes = 0;
    // multi-scan images (HJD_FLAG_MULTI_SCAN, csrc/multiscan.cu)
    std::vector<HjdScanDesc> scans;
    std::vector<HjdMsWork> mswork;              // one per (scan, restart interval), image order; sorted per chunk
    std::vector<uint32_t> ms_starts;            // interval starts of every scan (relative to the scan)
    std::vector<HjdHuffTable> ms_tabs;          // per-scan Huffman tables, de-duplicated by content
    std::unordered_multimap<uint64_t, uint32_t> ms_tab_of;
    std::vector<std::vector<uint8_t>> ms_tab_raw;
    std::vector<uint32_t> ms_items, n_scans;    // work items (multi-scan images), scans (0: not decodable)
    std::vector<uint8_t> ms_image;              // decoded by the multi-scan kernel (its blocks are zeroed first)
    // EXIF orientation.  orientation: what each file states (1..8), with or without the flag.  out_off: where each
    // image's output ends up in the slab, the offset every host consumer uses; it equals imgs[i].rgb_off unless the
    // image is oriented (HJD_FLAG_EXIF_ORIENT, orientation != 1), when imgs[i].rgb_off -- where the decode kernels write
    // -- is a private staging region of image_out_bytes behind rgb_bytes.  orient_jobs: one per oriented image, in
    // image order; orient_tiles: the exclusive prefix of their output tiles (n + 1).
    std::vector<uint8_t> orientation;
    std::vector<uint64_t> out_off;
    std::vector<HjdOrientJob> orient_jobs;
    std::vector<uint32_t> orient_tiles;
    uint64_t stage_bytes = 0;                   // staging regions, behind rgb_bytes in the same device allocation
    std::vector<Chunk> chunks;
    uint64_t total_blocks = 0, rgb_bytes = 0, plane_bytes = 0, scan_bytes = 0, pixels = 0;
    uint32_t total_intervals = 0;
    int max_tabs = 1;
    bool any_parse_error = false;
};

// Plans the upload of `files` (dev_off: each file's offset in the device arena) into *plan, which the caller has
// reset.  HJD_OK, or HJD_ERR_ARG with *err naming the index limit the batch would cross (DESIGN §3).
int hjd_plan_batch(const std::vector<FileRef>& files, const PlanConfig& cfg, BatchPlan* plan, std::string* err);
