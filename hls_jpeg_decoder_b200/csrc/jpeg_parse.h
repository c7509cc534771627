// csrc/jpeg_parse.h -- host side of the boundary: marker walk and table construction.
//
// Replaces the reference's "testbench" half (openjpg.cpp:371-496 ParseJFIF/JpegParseHeader,
// 120-155 DQT, 310-367 SOF, 234-305 DHT, 160-229 SOS, 48-98 canonical codes).  Unlike the
// reference it parses DRI properly (the reference stores Lr, openjpg.cpp:441-446), bounds
// every read, addresses components by position instead of id-as-index, and returns errors
// instead of printing and carrying on.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <vector>
#include "hjd_types.h"

struct HjdRawHuff {
    uint8_t present;
    uint8_t bits[16];
    uint8_t vals[256];
    int     nvals;
};

struct HjdParsed {
    int      status;             // HJD_IMG_* (0 = ok)
    uint32_t width, height;
    int      ncomp;              // 1 or 3
    int      hf, vf;             // luma sampling (1 for grayscale)
    int      tq[3], td[3], ta[3];
    uint8_t  qt[4][64];          // zig-zag order
    uint8_t  qt_present[4];
    HjdRawHuff dc[4], ac[4];
    uint32_t restart_interval;
    size_t   scan_off;           // offset of the first entropy-coded byte in the file
    size_t   scan_len;
    int      orientation;        // EXIF orientation 1..8 (1: none, or malformed; see hjd_exif_orientation)
};

// Header parse only (no table building).  Returns HJD_IMG_OK or a negative HJD_IMG_ERR_*.
int hjd_parse_jpeg(const uint8_t* buf, size_t size, HjdParsed* out);

// EXIF orientation of one APP1 payload (the bytes after the segment's length field, `len` of them): 0 when the payload
// does not start with "Exif\0\0" (not an Exif segment), else the value of IFD0's tag 0x0112 (type SHORT, count 1) in
// 1..8, or 1 when the TIFF structure is malformed, reaches past the payload, or has no such entry in IFD0.  Every read
// is bounded by `len`; no other IFD is followed.  Both marker walks take the first Exif APP1 before the first SOS.
int hjd_exif_orientation(const uint8_t* payload, size_t len);

// ---- multi-scan files (HJD_FLAG_MULTI_SCAN): progressive SOF2 and sequential files with several scans ----
struct HjdScanParsed {
    int      ncomp, comp[3];     // frame component indices, scan order
    int      ss, se, ah, al;
    int      kind, level;        // HJD_SCAN_* ; dependency level (see hjd_parse_jpeg_multi)
    uint32_t restart_interval;   // the DRI in effect at this scan (MCUs of this scan)
    size_t   off, len;           // entropy-coded segment in the file
    uint32_t first_start, n_starts;   // its RSTn-delimited interval starts (relative to off) in HjdMultiParsed::starts
    HjdRawHuff dc[3], ac[3];     // snapshot of the DHT contents this scan uses, per scan component (present = 0: unused)
};
struct HjdMultiParsed {
    HjdParsed frame;             // geometry and quantisation tables (Huffman fields unused)
    std::vector<HjdScanParsed> scans;
    std::vector<uint32_t> starts;
};

// Walk a whole file that hjd_parse_jpeg rejects as HJD_IMG_ERR_UNSUPPORTED and record every scan (T.81 G.1.1.1
// checked; scan headers that break it -> HJD_IMG_ERR_UNSUPPORTED).  A file that ends early keeps the scans it has.
// Each scan's end and RSTn positions are found by a host walk over its bytes.  Levels: 1 + the highest level of
// an earlier scan that shares a component and overlaps its band (DC = band {0}); 0 if none.  Scans of one level
// write disjoint (component, coefficient) positions.  Returns HJD_IMG_OK or a negative HJD_IMG_ERR_*.
int  hjd_parse_jpeg_multi(const uint8_t* buf, size_t size, HjdMultiParsed* out);
// Block grid of a scan: the frame's MCU grid when it is interleaved, the component's own block grid otherwise.
void hjd_scan_grid(const HjdParsed& f, const HjdScanParsed& s, uint32_t* mcus_x, uint32_t* mcus_y);

// Progressive AC tables: the same two-level lookup as hjd_build_huff_table, but each entry carries the raw
// run: len | size << 5 | run << 9 (EOBn keeps its n); HJD_BAD_ENTRY for no such code.
bool hjd_build_huff_table_raw(const HjdRawHuff& raw, HjdHuffTable* out);

// Length of the entropy-coded segment that starts at `scan` (avail bytes to the end of the file): up to
// the first marker that is neither FF00 nor RSTn (EOI normally).  Scans of HJD_SCAN_WALK_MAX bytes or
// more whose file ends with EOI are not walked.
#define HJD_SCAN_WALK_MAX (64u * 1024u)
size_t hjd_scan_length(const uint8_t* scan, size_t avail);

// Flattened lookup table from BITS/HUFFVAL.  Returns false if the code is over-subscribed.
bool hjd_build_huff_table(const HjdRawHuff& raw, bool is_ac, HjdHuffTable* out);

// Host mirror of the kernels' two-level symbol lookup: the entry for the next 16 bits (0: no such code).
uint32_t hjd_host_huff_lookup(const HjdHuffTable* t, uint32_t peek16);

// Resolve the per-component tables of a parsed image into a device table set / quant set.
// Returns HJD_IMG_OK or HJD_IMG_ERR_BAD_TABLE.
int hjd_build_table_set(const HjdParsed& p, HjdTableSet* out);
void hjd_build_quant_set(const HjdParsed& p, HjdQuantSet* out);

// The bytes a table set / quantisation set is built from, in canonical form (per component, in scan
// order: BITS + HUFFVAL of its DC and AC table; its quantisation table): equal bytes <=> equal sets.
struct HjdRawTables {
    uint8_t huff[4 + 3 * 2 * (16 + 256)];
    uint8_t quant[4 + 3 * 64];
};
void hjd_raw_tables(const HjdParsed& p, HjdRawTables* out);

// 64-bit content key of the tables an image uses (for sharing table sets across a batch).
uint64_t hjd_table_key(const HjdParsed& p);
uint64_t hjd_quant_key(const HjdParsed& p);

// Host RSTn scan (HJD_FLAG_HOST_SCAN and tests): writes the start offset (relative to the scan)
// of each restart interval; returns the number of intervals found (capped at max_out).
uint32_t hjd_host_find_intervals(const uint8_t* scan, size_t scan_len, uint32_t* starts, uint32_t max_out);
