// csrc/hjd_api.cu -- the C ABI of include/hjd.h: batch handle, HBM slabs, launches.
//
// Host-side counterpart of the reference's ConvertJpgFile / JpegDecodeHW call sequence
// (openjpg.cpp:593-684): load -> parse -> decode -> (write BMP).  Here "decode" is a set of
// kernel launches over flat HBM slabs holding N images, and nothing is decoded on the CPU.
#include "../../include/hjd.h"
#include "hjd_types.h"
#include "jpeg_parse.h"
#include "kernels.cuh"
#include "selfsync.cuh"
#include "multiscan.cuh"
#include "scaled.cuh"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <atomic>
#include <memory>
#include <string>
#include <thread>
#include <unordered_map>
#include <algorithm>
#include <vector>

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static_assert(HJD_MAX_SCANS == HJD_MAX_SCANS_PER_IMAGE, "hjd_types.h and include/hjd.h state the same scan cap");

static thread_local std::string g_err;

static int fail(int code, const char* what, const char* detail = nullptr)
{
    g_err = what;
    if (detail) { g_err += ": "; g_err += detail; }
    return code;
}

#define CU(call)                                                                     \
    do {                                                                             \
        cudaError_t e_ = (call);                                                     \
        if (e_ != cudaSuccess) return fail(HJD_ERR_CUDA, #call, cudaGetErrorString(e_)); \
    } while (0)

static inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------------------------------
// grow-only buffers
// ------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaError_t e = cudaFree(p); p = nullptr; cap = 0; if (e != cudaSuccess) return e; }
        size_t want = bytes + bytes / 16 + 4096;      // slack so that slowly growing batches do not reallocate
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); want = bytes; e = cudaMalloc(&p, want); }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocPortable);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// ------------------------------------------------------------------------------------------
// batch
// ------------------------------------------------------------------------------------------
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
    uint64_t blocks = 0;
    // kernel 1b (restart-free images of this chunk): ranges in the batch-wide index spaces, each with a gap of
    // one entry behind it so that the chunks' prefix sums (which append a sentinel) can run side by side
    uint32_t ss0 = 0, ss1 = 0;                // entries of b->ss
    uint32_t sub0 = 0, n_subs = 0;            // sub-sequences
    uint32_t ck0 = 0, n_ck = 0;               // 16-byte de-stuffing chunks
    uint32_t sw0 = 0, sw1 = 0, sf0 = 0, sf1 = 0;   // work items: speculative / write kernels, synchronisation kernel
    uint32_t ss_range = 0;                    // sub-sequences per warp in the synchronisation kernel
    // multi-scan images of this chunk: their slab blocks (zeroed before the first level), their work items per level
    std::vector<std::pair<uint64_t, uint64_t>> ms_zero;     // (first block, blocks)
    std::vector<std::pair<uint32_t, uint32_t>> ms_levels;   // work item range of each level present, in level order
};

#define HJD_NSTREAMS 3

struct hjd_batch {
    int device = 0;
    unsigned flags = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t mark[HJD_MARK_SLOTS] = {};                          // hjd_batch_mark
    cudaStream_t aux[HJD_NSTREAMS] = {nullptr, nullptr, nullptr}; // chunk streams
    cudaEvent_t ev_fork = nullptr, ev_join[HJD_NSTREAMS] = {nullptr, nullptr, nullptr};
    std::vector<Chunk> chunks;
    std::vector<FileRef> files;
    const uint8_t* contig_src = nullptr;      // host address of device-arena offset 0 (arena uploads)
    int overlap = 1;                                               // 0: one chunk, one stream (stage timings)
    int chunk_images = 0;                                          // > 0: images per chunk asked for by the caller of hjd_batch_decode_host

    // host metadata of the uploaded batch
    std::vector<HjdImageDesc> imgs;
    std::vector<int32_t> parse_status;
    std::vector<HjdTableSet> tsets;
    std::vector<HjdQuantSet> qsets;
    std::vector<HjdEntropyWork> work;
    std::vector<HjdEntropySeg> segs;
    std::vector<HjdScanSlice> slices;    // marker-scan slices of long restart-marker scans
    std::vector<uint32_t> mcu_cta;       // exclusive prefix of the per-image MCU counts (n + 1), for the flat grid of the per-MCU kernel
    std::vector<uint32_t> host_istart;          // HJD_FLAG_HOST_SCAN only
    std::vector<HjdSsImage> ss;                 // images on the self-synchronising path (kernel 1b)
    std::vector<HjdSsWork> sswork;       // one entry per CTA: speculative / write kernels, then synchronisation rounds
    std::vector<HjdSsSeg> sssegs;        // their segments
    uint32_t ss_range_req = 0;           // 0 = automatic
    uint32_t ss_subs = 0, ss_chunks = 0;          // batch-wide totals, including one gap per chunk
    uint32_t ss_tmp_stride = 0;                  // words of prefix-sum scratch per chunk
    uint64_t ss_dst_bytes = 0;
    bool ss_ran = false;                        // the last decode ran kernel 1b (its round count is in d_flag)
    int max_sync_ctas = 1;                      // grid limit of the cooperative synchronisation kernel on this device
    std::vector<uint8_t> host_restart_warn;     // HJD_FLAG_HOST_SCAN only (and multi-scan images)
    // multi-scan images (HJD_FLAG_MULTI_SCAN, csrc/multiscan.cu)
    std::vector<HjdScanDesc> scans;
    std::vector<HjdMsWork> mswork;              // one per (scan, restart interval), image order; sorted per chunk
    std::vector<uint32_t> ms_starts;            // interval starts of every scan (relative to the scan)
    std::vector<HjdHuffTable> ms_tabs;          // per-scan Huffman tables, de-duplicated by content
    std::unordered_multimap<uint64_t, uint32_t> ms_tab_of;
    std::vector<std::vector<uint8_t>> ms_tab_raw;
    std::vector<uint32_t> ms_items, n_scans;    // per image: work items (multi-scan images), scans (0: not decodable)
    std::vector<uint32_t> ms_w0;                // per image: its first work item (n + 1 entries)
    std::vector<uint8_t> ms_image;              // per image: decoded by the multi-scan kernel (its blocks are zeroed first)
    std::unordered_multimap<uint64_t, uint32_t> tset_of, qset_of;   // content hash -> candidate sets (verified byte for byte)
    std::vector<HjdRawTables> tset_raw, qset_raw;                    // what each set was built from
    uint64_t total_blocks = 0, rgb_bytes = 0, plane_bytes = 0, scan_bytes = 0, pixels = 0, arena_bytes = 0;
    uint32_t total_intervals = 0, max_blocks = 0, max_w = 0, max_h = 0;
    int max_tabs = 1;
    bool any_parse_error = false;
    bool uploaded = false, decoded = false;
    int launches = 0;
    int sm_count = 148;                         // multiprocessors of this device (work-list balancing)
    int tc_chunks = 0, cc_chunks = 0;           // chunks of the last decode whose MCUs went through the tensor-core / CUDA-core fused kernel
    int sc_chunks = 0;                          // ... through the scaled kernel (HJD_FLAG_SCALE_*)

    DevBuf d_arena, d_imgs, d_tsets, d_qsets, d_work, d_segs, d_mcucta, d_slices, d_slicecnt, d_istart, d_coef, d_planes, d_rgb, d_status;
    DevBuf d_scans, d_mswork, d_msstarts, d_mstabs;
    DevBuf d_ss, d_sswork, d_sssegs, d_destuff, d_dlen, d_counts, d_scantmp, d_ssE0, d_ssX, d_ssnb, d_flag;
    PinBuf h_meta, h_out;                       // h_out: staging of the single-image calls
};

// log2 of the scale denominator of HJD_FLAG_SCALE_* (0: full size), and the output size of a W x H image under it:
// ceil(W / d) x ceil(H / d), libjpeg's jdiv_round_up.
static int scale_shift(unsigned flags) { return (int)((flags & HJD_FLAG_SCALE_MASK) >> 9); }
static uint32_t scaled_dim(unsigned flags, uint32_t v)
{
    const int s = scale_shift(flags);
    return (uint32_t)(((uint64_t)v + (1u << s) - 1) >> s);
}

// Bytes of one image's region in the output slab: tightly packed RGB24 (of the scaled size with HJD_FLAG_SCALE_*), or
// (HJD_FLAG_BMP_OUT) the BMP file WriteBMP24 would write, placed so that its pixel array starts 64 bytes into the
// region (the 54-byte header at +10): rows padded to a multiple of 4 bytes, openjpg.cpp:534-535.
static uint64_t image_out_bytes(unsigned flags, uint32_t w, uint32_t h)
{
    if (flags & HJD_FLAG_BMP_OUT) return 64 + (uint64_t)((w * 3 + 3) & ~3u) * h;
    return (uint64_t)scaled_dim(flags, w) * scaled_dim(flags, h) * 3;
}

// The reduced IDCT's cosine table for N samples per block side: the expression of compute_idct_constants with 16
// replaced by 2N (host libm).
static void compute_scaled_cos(int n, float* cos_n)
{
    const float PI = 3.14f;
    for (int p = 0; p < n; p++)
        for (int k = 0; k < n; k++) cos_n[p * n + k] = cosf(((2 * p + 1) * k * PI) / (float)(2 * n));
}

static void compute_idct_constants(float cos_tab[64], float* cc0, float* cc00)
{
    // The very expressions of the reference, evaluated by the host libm (loadjpg.cpp:96-102,108,120).
    const float PI = 3.14f;
    for (int p = 0; p < 8; p++)
        for (int k = 0; k < 8; k++) cos_tab[p * 8 + k] = cosf(((2 * p + 1) * k * PI) / 16);
    volatile float c0 = 1.0f / sqrtf(2);
    *cc0 = c0 * 1.0f;
    *cc00 = c0 * c0;
}

extern "C" void hjd_get_idct_tables(float cos_tab[64], float cc[64])
{
    float c0, c00;
    compute_idct_constants(cos_tab, &c0, &c00);
    for (int u = 0; u < 8; u++)
        for (int v = 0; v < 8; v++) cc[u * 8 + v] = (u == 0 && v == 0) ? c00 : ((u == 0 || v == 0) ? c0 : 1.0f);
}

extern "C" void hjd_get_idct_matrix(uint16_t img[8192])
{
    float cos_tab[64], c0, c00;
    compute_idct_constants(cos_tab, &c0, &c00);
    hjd_build_idct_matrix(cos_tab, c0, c00, img);
}

extern "C" int hjd_version(void) { return HJD_VERSION; }
extern "C" const char* hjd_last_error(void) { return g_err.c_str(); }

extern "C" int hjd_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" hjd_batch* hjd_batch_create(int device, unsigned flags)
{
    int n = hjd_device_count();
    if (n <= 0) { fail(HJD_ERR_CUDA, "hjd_batch_create", "no CUDA device available (this library has no CPU fallback)"); return nullptr; }
    if (device < 0 || device >= n) { fail(HJD_ERR_ARG, "hjd_batch_create", "bad device index"); return nullptr; }
    if ((flags & HJD_FLAG_BMP_OUT) && (flags & HJD_FLAG_KEEP_PLANES)) { fail(HJD_ERR_ARG, "hjd_batch_create", "HJD_FLAG_BMP_OUT is an epilogue of the default (fused) kernels"); return nullptr; }
    if ((flags & HJD_FLAG_SCALE_MASK) &&
        (flags & (HJD_FLAG_KEEP_PLANES | HJD_FLAG_BMP_OUT | HJD_FLAG_TENSOR_CORE_IDCT | HJD_FLAG_CUDA_CORE_IDCT))) {
        fail(HJD_ERR_ARG, "hjd_batch_create", "HJD_FLAG_SCALE_* has no planes, no BMP output and its own kernel: it combines with "
                                              "none of HJD_FLAG_KEEP_PLANES, HJD_FLAG_BMP_OUT, HJD_FLAG_TENSOR_CORE_IDCT, HJD_FLAG_CUDA_CORE_IDCT");
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) { fail(HJD_ERR_CUDA, "cudaSetDevice"); return nullptr; }
    hjd_batch* b = new hjd_batch();
    b->device = device;
    b->flags = flags;
    cudaError_t e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
    b->own_stream = true;
    for (int i = 0; i < 5 && e == cudaSuccess; i++) e = cudaEventCreate(&b->ev[i]);
    for (int i = 0; i < HJD_MARK_SLOTS && e == cudaSuccess; i++) e = cudaEventCreate(&b->mark[i]);
    for (int i = 0; i < HJD_NSTREAMS && e == cudaSuccess; i++) e = cudaStreamCreateWithFlags(&b->aux[i], cudaStreamNonBlocking);
    for (int i = 0; i < HJD_NSTREAMS && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&b->ev_join[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = hjd_kernels_init_device();            // function attributes are per device
    if (e == cudaSuccess) e = hjd_selfsync_init_device(&b->max_sync_ctas);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&b->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) {
        float cos_tab[64], c0, c00;
        compute_idct_constants(cos_tab, &c0, &c00);
        e = hjd_set_idct_constants(cos_tab, c0, c00);
        if (e == cudaSuccess) {
            float cos4[16], cos2[4], cos1[1], cc[64], cc16[16];
            compute_scaled_cos(4, cos4);
            compute_scaled_cos(2, cos2);
            compute_scaled_cos(1, cos1);
            hjd_get_idct_tables(cos_tab, cc);
            for (int u = 0; u < 4; u++)
                for (int v = 0; v < 4; v++) cc16[u * 4 + v] = cc[u * 8 + v];
            e = hjd_set_scaled_constants(cos4, cos2, cos1, cc16);
        }
    }
    if (e != cudaSuccess) {
        fail(HJD_ERR_CUDA, "hjd_batch_create", cudaGetErrorString(e));
        hjd_batch_destroy(b);
        return nullptr;
    }
    return b;
}

extern "C" void hjd_batch_destroy(hjd_batch* b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->stream) cudaStreamSynchronize(b->stream);
    b->d_arena.release(); b->d_imgs.release(); b->d_tsets.release(); b->d_qsets.release(); b->d_work.release(); b->d_segs.release(); b->d_mcucta.release(); b->d_slices.release(); b->d_slicecnt.release();
    b->d_istart.release(); b->d_coef.release(); b->d_planes.release(); b->d_rgb.release(); b->d_status.release();
    b->d_ss.release(); b->d_sswork.release(); b->d_sssegs.release(); b->d_destuff.release(); b->d_dlen.release(); b->d_counts.release();
    b->d_scantmp.release(); b->d_ssE0.release(); b->d_ssX.release(); b->d_ssnb.release();
    b->d_flag.release();
    b->d_scans.release(); b->d_mswork.release(); b->d_msstarts.release(); b->d_mstabs.release();
    b->h_meta.release(); b->h_out.release();
    for (int i = 0; i < 5; i++) if (b->ev[i]) cudaEventDestroy(b->ev[i]);
    for (int i = 0; i < HJD_MARK_SLOTS; i++) if (b->mark[i]) cudaEventDestroy(b->mark[i]);
    for (int i = 0; i < HJD_NSTREAMS; i++) { if (b->aux[i]) { cudaStreamSynchronize(b->aux[i]); cudaStreamDestroy(b->aux[i]); } if (b->ev_join[i]) cudaEventDestroy(b->ev_join[i]); }
    if (b->ev_fork) cudaEventDestroy(b->ev_fork);
    if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
    delete b;
}

extern "C" int hjd_batch_set_stream(hjd_batch* b, void* cuda_stream)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_set_stream", "null batch");
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
    b->stream = (cudaStream_t)cuda_stream;
    b->own_stream = false;
    return HJD_OK;
}

// Index of the per-scan Huffman table built from `raw` (mode 0: DC, 1: sequential AC, 2: progressive AC with the raw
// run), shared by every scan of the batch with the same contents; -1: the code is over-subscribed.
static int ms_table(hjd_batch* b, const HjdRawHuff& raw, int mode)
{
    std::vector<uint8_t> key(17 + (size_t)raw.nvals);
    key[0] = (uint8_t)mode;
    memcpy(&key[1], raw.bits, 16);
    memcpy(&key[17], raw.vals, (size_t)raw.nvals);
    uint64_t h = 1469598103934665603ull;
    for (uint8_t v : key) { h ^= v; h *= 1099511628211ull; }
    auto range = b->ms_tab_of.equal_range(h);
    for (auto it = range.first; it != range.second; ++it)
        if (b->ms_tab_raw[it->second] == key) return (int)it->second;
    HjdHuffTable t;
    if (!(mode == 2 ? hjd_build_huff_table_raw(raw, &t) : hjd_build_huff_table(raw, mode == 1, &t))) return -1;
    b->ms_tabs.push_back(t);
    b->ms_tab_raw.push_back(std::move(key));
    b->ms_tab_of.emplace(h, (uint32_t)b->ms_tabs.size() - 1);
    return (int)b->ms_tabs.size() - 1;
}

// Work items of one scan: the restart intervals its DRI implies (want_all) or, by default, no more than the file holds.
static uint32_t ms_scan_items(const HjdParsed& frame, const HjdScanParsed& p, uint32_t* mcus_x, uint32_t* mcus_y,
                              bool want_all = false)
{
    uint32_t mx, my;
    hjd_scan_grid(frame, p, &mx, &my);
    if (mcus_x) { *mcus_x = mx; *mcus_y = my; }
    const uint64_t total = (uint64_t)mx * my;
    const uint64_t want = p.restart_interval ? (total + p.restart_interval - 1) / p.restart_interval : 1;
    return (uint32_t)(want_all || want < p.n_starts ? want : p.n_starts);
}

// Scan descriptors, tables, interval starts and work items of multi-scan image i (file at arena offset dev_off).
// A scan with fewer RSTn markers than its DRI implies (a file cut inside it) gets the intervals it has: the last one
// runs to the end of the data, and the image is flagged HJD_IMG_WARN_RESTART.  HJD_IMG_OK or HJD_IMG_ERR_BAD_TABLE.
static int ms_add_image(hjd_batch* b, int i, const HjdMultiParsed& mp, uint64_t dev_off)
{
    const size_t scan0 = b->scans.size(), start0 = b->ms_starts.size(), work0 = b->mswork.size();
    uint32_t items = 0, n_scans = 0;
    // At 1/8 a block is its DC coefficient alone: the AC scans (Ss > 0) are not read.
    const bool dc_only = scale_shift(b->flags) == 3;
    for (const HjdScanParsed& p : mp.scans) {
        if (dc_only && p.ss > 0) continue;
        n_scans++;
        HjdScanDesc sd;
        memset(&sd, 0, sizeof sd);
        sd.image = (uint32_t)i;
        sd.ncomp = (uint8_t)p.ncomp;
        for (int k = 0; k < p.ncomp; k++) sd.comp[k] = (uint8_t)p.comp[k];
        sd.ss = (uint8_t)p.ss; sd.se = (uint8_t)p.se; sd.ah = (uint8_t)p.ah; sd.al = (uint8_t)p.al;
        sd.kind = (uint8_t)p.kind; sd.level = (uint8_t)(p.level < 255 ? p.level : 255);
        sd.restart_interval = p.restart_interval;
        sd.n_intervals = ms_scan_items(mp.frame, p, &sd.mcus_x, &sd.mcus_y);
        if (p.restart_interval && p.n_starts != ms_scan_items(mp.frame, p, nullptr, nullptr, true)) b->host_restart_warn[i] = 1;
        sd.start_base = (uint32_t)b->ms_starts.size();
        sd.scan_len = (uint32_t)p.len;
        sd.scan_off = dev_off + p.off;
        for (int k = 0; k < p.ncomp; k++) {
            const int td = p.dc[k].present ? ms_table(b, p.dc[k], 0) : 0;
            const int ta = p.ac[k].present ? ms_table(b, p.ac[k], p.kind == HJD_SCAN_SEQ ? 1 : 2) : 0;
            if (td < 0 || ta < 0) {
                b->scans.resize(scan0); b->ms_starts.resize(start0); b->mswork.resize(work0);
                return HJD_IMG_ERR_BAD_TABLE;
            }
            sd.dc_tab[k] = (uint32_t)td;
            sd.ac_tab[k] = (uint32_t)ta;
        }
        for (uint32_t j = 0; j < sd.n_intervals; j++) {
            b->ms_starts.push_back(mp.starts[p.first_start + j]);
            b->mswork.push_back(HjdMsWork{(uint32_t)b->scans.size(), j});
        }
        items += sd.n_intervals;
        b->scans.push_back(sd);
    }
    b->ms_items[i] = items;
    b->n_scans[i] = n_scans;
    return HJD_OK;
}

// Parse + lay out + upload the metadata.  b->files[i].dev_off must already hold the arena offset of
// file i.  The files themselves are copied by copy_files(), whole or chunk by chunk.
static int upload_common(hjd_batch* b, bool chunked)
{
    std::vector<FileRef>& files = b->files;
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));     // staging buffers of the previous batch are free again
    const int n = (int)files.size();
    b->chunks.clear();
    b->imgs.assign(n, HjdImageDesc());
    b->parse_status.assign(n, 0);
    b->tsets.clear(); b->qsets.clear(); b->tset_of.clear(); b->qset_of.clear(); b->tset_raw.clear(); b->qset_raw.clear(); b->work.clear(); b->segs.clear(); b->slices.clear();
    b->host_istart.clear();
    b->host_restart_warn.assign(n, 0);
    b->ss.clear(); b->sswork.clear(); b->sssegs.clear();
    b->scans.clear(); b->mswork.clear(); b->ms_starts.clear(); b->ms_tabs.clear(); b->ms_tab_of.clear(); b->ms_tab_raw.clear();
    b->ms_items.assign(n, 0); b->n_scans.assign(n, 0); b->ms_w0.assign((size_t)n + 1, 0); b->ms_image.assign(n, 0);
    b->ss_subs = b->ss_chunks = 0;
    b->ss_dst_bytes = 0;
    b->total_blocks = b->rgb_bytes = b->plane_bytes = b->scan_bytes = b->pixels = 0;
    b->total_intervals = b->max_blocks = b->max_w = b->max_h = 0;
    b->max_tabs = 1;
    b->any_parse_error = false;
    b->uploaded = b->decoded = false;

    // Header parse and table hashing of every image, in parallel for large batches (8192 thumbnails: 9 ms
    // of the host's time on one thread).  What the serial pass below needs is kept in a small record;
    // the few images that bring a new table or quantisation set are parsed once more there.
    // Table and quantisation sets are shared by images with identical DHT / DQT contents.  The 64-bit
    // hash only finds candidates: every worker keeps the raw tables of the images that introduced a key
    // (to that worker) and compares the bytes on a hit, so an image is either byte-identical to an earlier
    // image of its worker (trep / qrep = that image) or a representative itself; representatives are
    // compared byte for byte with the sets built so far in the serial pass.  A hash collision therefore
    // costs a set of its own, never somebody else's tables.
    struct Lite {
        int status;
        uint32_t width, height, restart_interval;
        int ncomp, hf, vf;
        size_t scan_off, scan_len;
        uint64_t tk, qk;
        uint64_t ms_items;         // multi-scan work items (what ms_add_image will add)
        int trep, qrep;            // image whose tables / quantisation tables these are byte-identical to (itself: a representative)
    };
    std::vector<Lite> lite((size_t)n);
    // HJD_FLAG_MULTI_SCAN: files the single-scan parse rejects as unsupported get the multi-scan walk; these
    // images keep the result (scans, interval starts, table snapshots) for the serial pass
    std::vector<std::unique_ptr<HjdMultiParsed>> multi((size_t)n);
    auto parse_range = [&](int lo, int hi) {
        HjdParsed p;
        struct Seen { uint64_t key; int image; HjdRawTables raw; };
        std::vector<Seen> seen_t, seen_q;
        HjdRawTables raw;
        for (int i = lo; i < hi; i++) {
            Lite& l = lite[(size_t)i];
            memset(&l, 0, sizeof l);
            int st = (files[i].ptr && files[i].size > 0) ? hjd_parse_jpeg(files[i].ptr, (size_t)files[i].size, &p)
                                                         : HJD_IMG_ERR_NOT_JPEG;
            if (st == HJD_IMG_OK && p.scan_len > 0xFFFFFF00ull) st = HJD_IMG_ERR_UNSUPPORTED;
            if (st == HJD_IMG_ERR_UNSUPPORTED && (b->flags & HJD_FLAG_MULTI_SCAN)) {
                std::unique_ptr<HjdMultiParsed> mp(new HjdMultiParsed());
                st = hjd_parse_jpeg_multi(files[i].ptr, (size_t)files[i].size, mp.get());
                if (st == HJD_IMG_OK && mp->frame.scan_len > 0xFFFFFF00ull) st = HJD_IMG_ERR_UNSUPPORTED;
                if (st == HJD_IMG_OK) {
                    p = mp->frame;
                    for (const HjdScanParsed& sp : mp->scans)
                        if (!(scale_shift(b->flags) == 3 && sp.ss > 0)) l.ms_items += ms_scan_items(mp->frame, sp, nullptr, nullptr);
                    multi[(size_t)i] = std::move(mp);
                }
            }
            l.status = st;
            if (st != HJD_IMG_OK) continue;
            l.width = p.width; l.height = p.height; l.restart_interval = p.restart_interval;
            l.ncomp = p.ncomp; l.hf = p.hf; l.vf = p.vf;
            l.scan_off = p.scan_off; l.scan_len = p.scan_len;
            l.tk = hjd_table_key(p); l.qk = hjd_quant_key(p);
            hjd_raw_tables(p, &raw);
            l.trep = l.qrep = i;
            bool hit = multi[(size_t)i] != nullptr;      // multi-scan images carry per-scan tables instead of a table set
            for (const Seen& sn : seen_t)
                if (sn.key == l.tk && memcmp(sn.raw.huff, raw.huff, sizeof raw.huff) == 0) { l.trep = sn.image; hit = true; break; }
            if (!hit && seen_t.size() < 64) seen_t.push_back(Seen{l.tk, i, raw});
            if (multi[(size_t)i]) hit = false;
            hit = false;
            for (const Seen& sn : seen_q)
                if (sn.key == l.qk && memcmp(sn.raw.quant, raw.quant, sizeof raw.quant) == 0) { l.qrep = sn.image; hit = true; break; }
            if (!hit && seen_q.size() < 64) seen_q.push_back(Seen{l.qk, i, raw});
        }
    };
    {
        unsigned hw = std::thread::hardware_concurrency();
        int nt = n >= 2048 ? (int)(hw < 2 ? 1 : (hw > 8 ? 8 : hw)) : 1;
        if (nt <= 1) parse_range(0, n);
        else {
            std::vector<std::thread> pool;
            const int per = (n + nt - 1) / nt;
            for (int k = 0; k < nt; k++) {
                const int lo = k * per, hi = lo + per < n ? lo + per : n;
                if (lo < hi) pool.emplace_back(parse_range, lo, hi);
            }
            for (auto& th : pool) th.join();
        }
    }

    // Index limits a batch must stay inside (DESIGN §3), refused before anything is allocated or copied.  Multi-scan
    // work items are numbered in int (hjd_k_multiscan's thread index), so a batch holds fewer than 2^31.
    {
        uint64_t items = 0;
        for (const Lite& l : lite) items += l.ms_items;
        if (items >= 0x80000000ull) return fail(HJD_ERR_ARG, "hjd_batch_upload", "batch exceeds 2^31 multi-scan work items");
    }

    HjdParsed full;                    // re-parse target for the representatives
    HjdRawTables full_raw;
    std::vector<uint32_t> tset_of_img((size_t)n, 0), qset_of_img((size_t)n, 0);
    for (int i = 0; i < n; i++) {
        HjdImageDesc& d = b->imgs[i];
        memset(&d, 0, sizeof d);
        d.interval_base = b->total_intervals;
        d.block_base = b->total_blocks;
        d.rgb_off = b->rgb_bytes;
        d.y_off = d.cb_off = d.cr_off = b->plane_bytes;
        const Lite& ps = lite[(size_t)i];
        int st = ps.status;
        uint32_t tset = 0, qset = 0;
        bool have_full = false;
        const HjdMultiParsed* mp = multi[(size_t)i].get();
        if (st == HJD_IMG_OK && mp) {
            st = ms_add_image(b, i, *mp, files[i].dev_off);
            b->ms_image[i] = 1;
            full = mp->frame;
            hjd_raw_tables(full, &full_raw);
            have_full = true;
        } else if (st == HJD_IMG_OK) {
            if (ps.trep != i) {                                     // byte-identical to an earlier image of its worker
                if (b->parse_status[ps.trep] != HJD_IMG_OK) st = b->parse_status[ps.trep];      // e.g. an over-subscribed DHT
                tset = tset_of_img[(size_t)ps.trep];
            } else {
                hjd_parse_jpeg(files[i].ptr, (size_t)files[i].size, &full);
                hjd_raw_tables(full, &full_raw);
                have_full = true;
                bool found = false;
                auto range = b->tset_of.equal_range(ps.tk);
                for (auto it = range.first; it != range.second && !found; ++it)
                    if (memcmp(b->tset_raw[it->second].huff, full_raw.huff, sizeof full_raw.huff) == 0) { tset = it->second; found = true; }
                if (!found) {
                    HjdTableSet ts;
                    st = hjd_build_table_set(full, &ts);
                    if (st == HJD_IMG_OK) {
                        tset = (uint32_t)b->tsets.size(); b->tsets.push_back(ts); b->tset_raw.push_back(full_raw);
                        b->tset_of.emplace(ps.tk, tset);
                        if (ts.n_tabs > b->max_tabs) b->max_tabs = ts.n_tabs;
                    }
                }
            }
        }
        if (st == HJD_IMG_OK) {
            if (ps.qrep != i) qset = qset_of_img[(size_t)ps.qrep];
            else {
                if (!have_full) { hjd_parse_jpeg(files[i].ptr, (size_t)files[i].size, &full); hjd_raw_tables(full, &full_raw); }
                bool found = false;
                auto range = b->qset_of.equal_range(ps.qk);
                for (auto it = range.first; it != range.second && !found; ++it)
                    if (memcmp(b->qset_raw[it->second].quant, full_raw.quant, sizeof full_raw.quant) == 0) { qset = it->second; found = true; }
                if (!found) {
                    HjdQuantSet qs;
                    hjd_build_quant_set(full, &qs);
                    qset = (uint32_t)b->qsets.size(); b->qsets.push_back(qs); b->qset_raw.push_back(full_raw);
                    b->qset_of.emplace(ps.qk, qset);
                }
            }
        }
        tset_of_img[(size_t)i] = tset; qset_of_img[(size_t)i] = qset;
        b->parse_status[i] = st;
        b->ms_w0[(size_t)i + 1] = (uint32_t)b->mswork.size();
        if (st != HJD_IMG_OK) { b->any_parse_error = true; continue; }   // n_intervals = n_blocks = 0: skipped
        if (!mp) b->n_scans[i] = 1;

        d.width = ps.width; d.height = ps.height;
        d.ncomp = (uint8_t)ps.ncomp; d.hf = (uint8_t)ps.hf; d.vf = (uint8_t)ps.vf;
        d.blocks_per_mcu = (uint8_t)(ps.ncomp == 3 ? ps.hf * ps.vf + 2 : 1);
        d.mcus_x = (ps.width + 8 * ps.hf - 1) / (8 * ps.hf);            // loadjpg.cpp:1170-1174
        d.mcus_y = (ps.height + 8 * ps.vf - 1) / (8 * ps.vf);
        d.n_mcus = d.mcus_x * d.mcus_y;
        d.restart_interval = ps.restart_interval;
        d.n_intervals = ps.restart_interval ? (d.n_mcus + ps.restart_interval - 1) / ps.restart_interval : 1;
        d.scan_len = (uint32_t)ps.scan_len;
        d.scan_off = files[i].dev_off + ps.scan_off;
        if (mp) d.n_intervals = 0;                   // entropy decode by the multi-scan kernel only (no kernel 0 / 1a / 1b)
        if (!mp && !(b->flags & HJD_FLAG_NO_SELFSYNC) && ps.restart_interval == 0 && ps.scan_len >= HJD_SS_MIN_BYTES) {
            // restart-free scan: kernel 1b (speculative self-synchronising decode) instead of one thread
            HjdSsImage si;
            memset(&si, 0, sizeof si);
            si.img = (uint32_t)i;
            si.n_subs = (uint32_t)((ps.scan_len + HJD_SS_SUB_BYTES - 1) / HJD_SS_SUB_BYTES);
            si.lead = (uint32_t)(d.scan_off & 15);
            si.n_chunks = (uint32_t)((ps.scan_len + si.lead + 15) / 16);
            si.dst_off = b->ss_dst_bytes;
            d.n_intervals = 0;
            d.n_subs = si.n_subs;
            b->ss.push_back(si);                 // sub_base / chunk_base: after the chunk plan (below)
            b->ss_dst_bytes += align_up(ps.scan_len + HJD_SS_SLACK + 16, 256);   // + 16: the slack is zeroed from the next 16-byte boundary
        }
        d.table_set = tset; d.quant_set = qset;
        d.n_blocks = (uint64_t)d.n_mcus * d.blocks_per_mcu;
        d.y_pitch = d.mcus_x * 8 * ps.hf;
        d.c_pitch = d.mcus_x * 8;
        const uint64_t ysz = (uint64_t)d.y_pitch * d.mcus_y * 8 * ps.vf;
        const uint64_t csz = ps.ncomp == 3 ? (uint64_t)d.c_pitch * d.mcus_y * 8 : 0;
        d.y_off = b->plane_bytes;
        d.cb_off = d.y_off + align_up(ysz, 256);
        d.cr_off = d.cb_off + align_up(csz, 256);
        b->plane_bytes = d.cr_off + align_up(csz, 256);
        b->rgb_bytes += align_up(image_out_bytes(b->flags, ps.width, ps.height), 256);
        b->total_intervals += d.n_intervals;
        b->total_blocks += d.n_blocks;
        b->scan_bytes += ps.scan_len;
        b->pixels += (uint64_t)ps.width * ps.height;
        if (d.n_blocks > b->max_blocks) b->max_blocks = (uint32_t)d.n_blocks;
        if (ps.width > b->max_w) b->max_w = ps.width;
        if (ps.height > b->max_h) b->max_h = ps.height;

        if ((b->flags & HJD_FLAG_HOST_SCAN) && d.n_intervals) {
            const size_t at = b->host_istart.size();
            b->host_istart.resize(at + d.n_intervals, (uint32_t)ps.scan_len);
            const uint32_t found = hjd_host_find_intervals(files[i].ptr + ps.scan_off, ps.scan_len,
                                                           b->host_istart.data() + at, d.n_intervals);
            if (ps.restart_interval && found != d.n_intervals) b->host_restart_warn[i] = 1;
        }
    }
    if (b->total_blocks >= 0xFFFFFFFFull) return fail(HJD_ERR_ARG, "hjd_batch_upload", "batch exceeds 2^32 blocks");
    {
        // kernel 1b numbers the 16-byte chunks of the restart-free scans in uint32, with one gap per chunk of the plan and
        // a sentinel: about 64 GiB of restart-free scan data
        uint64_t ck = 0;
        for (const HjdSsImage& si : b->ss) ck += si.n_chunks;
        if (ck + (uint64_t)n + 2 > 0xFFFFFFFFull)
            return fail(HJD_ERR_ARG, "hjd_batch_upload", "restart-free scans of the batch exceed 2^32 16-byte chunks (64 GiB)");
    }

    // chunk plan: contiguous image ranges of roughly equal block counts
    {
        int want = 1;
        if (chunked && b->overlap) {
            const uint64_t per_chunk = b->overlap > 1 ? (uint64_t)b->overlap : 1500000ull;
            want = (int)(b->total_blocks / per_chunk);
            if (want > 8) want = 8;
            if (want > n) want = n;
            if (want < 1) want = 1;
        }
        const uint64_t target = (b->total_blocks + want - 1) / (uint64_t)want;
        const int per = (chunked && b->chunk_images > 0) ? b->chunk_images : 0;   // caller-chosen chunk length (hjd_batch_decode_host)
        Chunk c;
        c.img0 = 0;
        for (int i = 0; i < n; i++) {
            c.blocks += b->imgs[i].n_blocks;
            const bool last = (i == n - 1);
            if (last || (per ? (i + 1 - c.img0 >= per) : (c.blocks >= target && (int)b->chunks.size() < want - 1))) {
                c.img1 = i + 1;
                b->chunks.push_back(c);
                c = Chunk();
                c.img0 = i + 1;
            }
        }
        if (n == 0) b->chunks.clear();
    }
    // per chunk: extents, grid bounds and the entropy work list (never crossing a chunk boundary)
    for (Chunk& c : b->chunks) {
        c.work0 = (uint32_t)b->work.size();
        c.arena_lo = ~0ull; c.arena_hi = 0;
        c.rgb_lo = b->imgs[c.img0].rgb_off;
        c.rgb_hi = (c.img1 < n) ? b->imgs[c.img1].rgb_off : b->rgb_bytes;
        for (int i = c.img0; i < c.img1; i++) {
            const HjdImageDesc& d = b->imgs[i];
            if (files[i].ptr && files[i].size > 0) {
                if (files[i].dev_off < c.arena_lo) c.arena_lo = files[i].dev_off;
                if (files[i].dev_off + (uint64_t)files[i].size > c.arena_hi) c.arena_hi = files[i].dev_off + (uint64_t)files[i].size;
            }
            if (d.n_blocks > c.max_blocks) c.max_blocks = (uint32_t)d.n_blocks;
            if (d.n_mcus > c.max_mcus) c.max_mcus = d.n_mcus;
            if (d.width > c.max_w) c.max_w = d.width;
            if (d.height > c.max_h) c.max_h = d.height;
        }
        // marker-scan slices of long restart-marker scans (kernel 0)
        c.slice0 = (uint32_t)b->slices.size();
        for (int i = c.img0; i < c.img1; i++) {
            const HjdImageDesc& d = b->imgs[i];
            if (d.restart_interval && d.n_intervals > 1 && d.scan_len > HJD_SCAN_SLICE_MIN) {
                const uint64_t total = (uint64_t)d.scan_len + (d.scan_off & 15);
                const uint32_t ns = (uint32_t)((total + HJD_SCAN_SLICE_BYTES - 1) / HJD_SCAN_SLICE_BYTES);
                for (uint32_t k = 0; k < ns; k++) b->slices.push_back(HjdScanSlice{(uint32_t)i, k, ns, 0});
            }
        }
        c.slice1 = (uint32_t)b->slices.size();
        // entropy work items: the chunk's images grouped by table set (batch order kept inside a group),
        // their intervals packed into CTAs of HJD_ENT_THREADS as segments
        {
            std::vector<int> order;
            for (int i = c.img0; i < c.img1; i++) if (b->imgs[i].n_intervals) order.push_back(i);
            std::stable_sort(order.begin(), order.end(),
                             [&](int x, int y) { return b->imgs[x].table_set < b->imgs[y].table_set; });
            // Intervals per CTA.  A big chunk fills its CTAs (HJD_ENT_THREADS).  A chunk of only a few waves -- one 1024-image
            // batch cut over 8 GPUs is 0.86 of a wave -- is cut into a whole number of waves of equally loaded CTAs instead:
            // with 510 full CTAs on 592 slots the SMs that got four of them set the time; 592 CTAs of 221 intervals finish
            // in 0.86 of it.  (Below half a wave the CTAs stay full: fewer table loads, and nothing to balance.)
            uint32_t cap = HJD_ENT_THREADS;
            {
                uint64_t total = 0;
                for (int i : order) total += b->imgs[i].n_intervals;
                const uint64_t slots = (uint64_t)b->sm_count * HJD_ENT_MINBLOCKS;
                const uint64_t full = (total + HJD_ENT_THREADS - 1) / HJD_ENT_THREADS;
                if (2 * full >= slots && full <= 4 * slots) {
                    const uint64_t n_ctas = (full + slots - 1) / slots * slots;
                    cap = (uint32_t)((total + n_ctas - 1) / n_ctas);
                    if (cap > HJD_ENT_THREADS) cap = HJD_ENT_THREADS;
                    if (cap < 32) cap = 32;
                }
            }
            HjdEntropyWork w{0, 0, 0, 0};
            auto flush = [&]() {
                if (w.n_intervals) b->work.push_back(w);
                w = HjdEntropyWork{(uint32_t)b->segs.size(), 0, 0, 0};
            };
            flush();
            for (int i : order) {
                const HjdImageDesc& d = b->imgs[i];
                if (w.n_intervals && w.table_set != d.table_set) flush();
                uint32_t left = d.n_intervals, g = d.interval_base;
                while (left) {
                    if (w.n_intervals == cap) flush();
                    w.table_set = d.table_set;
                    const uint32_t take = left < (cap - w.n_intervals) ? left : (cap - w.n_intervals);
                    b->segs.push_back(HjdEntropySeg{g, w.n_intervals, (uint32_t)i, take});
                    w.n_segs++;
                    w.n_intervals += take; g += take; left -= take;
                }
            }
            if (w.n_intervals) b->work.push_back(w);
        }
        c.work1 = (uint32_t)b->work.size();
        if (c.arena_lo == ~0ull) c.arena_lo = c.arena_hi = 0;
        // multi-scan work of the chunk: by level (one launch each), then by kind, so that the lanes of a warp mostly run
        // the same loop.  A counting sort: a comparison sort of the 30 M items of 1024 1080p files with restart markers
        // every 8 blocks took seconds of host time.
        {
            const uint32_t w0 = b->ms_w0[(size_t)c.img0], w1 = b->ms_w0[(size_t)c.img1];
            std::vector<uint32_t> at(256 * 5 + 1, 0);
            for (uint32_t k = w0; k < w1; k++) {
                const HjdScanDesc& sd = b->scans[b->mswork[k].scan];
                at[sd.level * 5u + sd.kind + 1]++;
            }
            for (size_t q = 1; q < at.size(); q++) at[q] += at[q - 1];
            std::vector<HjdMsWork> sorted(w1 - w0);
            for (uint32_t k = w0; k < w1; k++) {
                const HjdScanDesc& sd = b->scans[b->mswork[k].scan];
                sorted[at[sd.level * 5u + sd.kind]++] = b->mswork[k];
            }
            std::copy(sorted.begin(), sorted.end(), b->mswork.begin() + w0);
            for (uint32_t k = w0; k < w1;) {
                const uint8_t lv = b->scans[b->mswork[k].scan].level;
                uint32_t e = k;
                while (e < w1 && b->scans[b->mswork[e].scan].level == lv) e++;
                c.ms_levels.emplace_back(k, e);
                k = e;
            }
            for (int i = c.img0; i < c.img1; i++) {
                if (!b->ms_image[i] || b->parse_status[i] != HJD_IMG_OK) continue;
                const HjdImageDesc& d = b->imgs[i];
                if (!c.ms_zero.empty() && c.ms_zero.back().first + c.ms_zero.back().second == d.block_base)
                    c.ms_zero.back().second += d.n_blocks;
                else
                    c.ms_zero.emplace_back(d.block_base, d.n_blocks);
            }
        }
    }

    // device slabs
    CU(b->d_arena.ensure(b->arena_bytes + 64));
    CU(b->d_imgs.ensure(sizeof(HjdImageDesc) * (size_t)(n + 1)));
    CU(b->d_tsets.ensure(sizeof(HjdTableSet) * (b->tsets.size() + 1)));
    CU(b->d_qsets.ensure(sizeof(HjdQuantSet) * (b->qsets.size() + 1)));
    CU(b->d_work.ensure(sizeof(HjdEntropyWork) * (b->work.size() + 1)));
    CU(b->d_segs.ensure(sizeof(HjdEntropySeg) * (b->segs.size() + 1)));
    CU(b->d_slices.ensure(sizeof(HjdScanSlice) * (b->slices.size() + 1)));
    CU(b->d_slicecnt.ensure(sizeof(uint32_t) * (b->slices.size() + 1)));
    b->mcu_cta.assign((size_t)n + 1, 0);
    for (int i = 0; i < n; i++)
        b->mcu_cta[i + 1] = b->mcu_cta[i] + (b->imgs[i].blocks_per_mcu ? b->imgs[i].n_mcus : 0);
    CU(b->d_mcucta.ensure(sizeof(uint32_t) * ((size_t)n + 2)));
    CU(b->d_istart.ensure(sizeof(uint32_t) * ((size_t)b->total_intervals + 2)));
    CU(b->d_coef.ensure(b->total_blocks * 128 + 256));
    CU(b->d_rgb.ensure(b->rgb_bytes + 256));
    CU(b->d_status.ensure(sizeof(int32_t) * (size_t)(n + 1)));
    if (b->flags & HJD_FLAG_KEEP_PLANES) CU(b->d_planes.ensure(b->plane_bytes + 256));
    // Kernel 1b, chunk by chunk (so that restart-free images pipeline like the rest: nothing in it needs the
    // host any more).  Index spaces are batch-wide with one spare entry after every chunk.  Inside a chunk the
    // images are grouped by table set (batch order kept inside a group) and their sub-sequences packed into
    // CTAs as segments, so small restart-free images share CTAs.  Synchronisation kernel: one range per warp;
    // longer ranges make the re-decode lists denser, shorter ones give more independent warps: by the amount
    // of work in the chunk.
    {
        size_t k0 = 0;
        uint32_t max_scan = 0;
        for (Chunk& c : b->chunks) {
            c.ss0 = (uint32_t)k0;
            c.sub0 = b->ss_subs;
            c.ck0 = b->ss_chunks;
            while (k0 < b->ss.size() && (int)b->ss[k0].img < c.img1) {
                HjdSsImage& si = b->ss[k0++];
                si.sub_base = b->ss_subs;
                si.chunk_base = b->ss_chunks;
                b->imgs[si.img].sub_base = si.sub_base;
                b->ss_subs += si.n_subs;
                b->ss_chunks += si.n_chunks;
            }
            c.ss1 = (uint32_t)k0;
            c.n_subs = b->ss_subs - c.sub0;
            c.n_ck = b->ss_chunks - c.ck0;
            b->ss_subs += 1;                     // the gaps
            b->ss_chunks += 1;
            if (c.n_ck + 1 > max_scan) max_scan = c.n_ck + 1;
            if (4 * c.n_subs + 2 > max_scan) max_scan = 4 * c.n_subs + 2;

            std::vector<uint32_t> order;
            for (uint32_t k = c.ss0; k < c.ss1; k++) order.push_back(k);
            std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) {
                return b->imgs[b->ss[x].img].table_set < b->imgs[b->ss[y].img].table_set;
            });
            HjdSsWork w{0, 0, 0, 0};
            auto flush = [&]() {
                if (w.n_subs) b->sswork.push_back(w);
                w = HjdSsWork{(uint32_t)b->sssegs.size(), 0, 0, 0};
            };
            flush();
            c.sw0 = (uint32_t)b->sswork.size();
            for (uint32_t k : order) {
                const uint32_t ts = b->imgs[b->ss[k].img].table_set;
                if (w.n_subs && w.table_set != ts) flush();
                uint32_t left = b->ss[k].n_subs, f = 0;
                while (left) {
                    if (w.n_subs == HJD_SS_THREADS) flush();
                    w.table_set = ts;
                    const uint32_t take = left < (HJD_SS_THREADS - w.n_subs) ? left : (HJD_SS_THREADS - w.n_subs);
                    b->sssegs.push_back(HjdSsSeg{k, f, w.n_subs, take});
                    w.n_segs++; w.n_subs += take; f += take; left -= take;
                }
            }
            flush();
            c.sw1 = c.sf0 = (uint32_t)b->sswork.size();
            c.ss_range = b->ss_range_req ? b->ss_range_req : c.n_subs >= 400000 ? 256 : c.n_subs >= 150000 ? 128 : 64;
            if (!b->ss_range_req && HJD_SS_FIX_MAXR >= 512 && c.n_subs >= 1000000) c.ss_range = 512;
            for (uint32_t k : order) {
                const uint32_t ts = b->imgs[b->ss[k].img].table_set;
                for (uint32_t f = 0; f < b->ss[k].n_subs; f += c.ss_range) {
                    if (w.n_segs == HJD_SS_FIX_WARPS || (w.n_segs && w.table_set != ts)) flush();
                    w.table_set = ts;
                    const uint32_t take = b->ss[k].n_subs - f < c.ss_range ? b->ss[k].n_subs - f : c.ss_range;
                    b->sssegs.push_back(HjdSsSeg{k, f, 0, take});
                    w.n_segs++; w.n_subs += take;
                }
            }
            flush();
            c.sf1 = (uint32_t)b->sswork.size();
        }
        b->ss_tmp_stride = max_scan / 2048 + 8;
    }

    if (!b->ss.empty()) {
        CU(b->d_ss.ensure(sizeof(HjdSsImage) * b->ss.size()));
        CU(b->d_sswork.ensure(sizeof(HjdSsWork) * b->sswork.size()));
        CU(b->d_sssegs.ensure(sizeof(HjdSsSeg) * (b->sssegs.size() + 1)));
        CU(b->d_destuff.ensure(b->ss_dst_bytes + 256));
        CU(b->d_dlen.ensure(sizeof(uint32_t) * b->ss.size()));
        CU(b->d_counts.ensure(sizeof(uint32_t) * ((size_t)b->ss_chunks + 2)));
        CU(b->d_scantmp.ensure(sizeof(uint32_t) * (size_t)b->ss_tmp_stride * (b->chunks.size() + 1)));
        CU(b->d_ssE0.ensure(sizeof(uint64_t) * (size_t)b->ss_subs));
        CU(b->d_ssX.ensure(sizeof(uint64_t) * (size_t)b->ss_subs));
        CU(b->d_ssnb.ensure(sizeof(uint32_t) * (4 * (size_t)b->ss_subs + 4)));
        CU(b->d_flag.ensure(sizeof(uint32_t) * 4 * (b->chunks.size() + 1)));
    }

    // metadata: one pinned staging block, then async copies
    const size_t sz_imgs = sizeof(HjdImageDesc) * (size_t)n;
    const size_t sz_ts = sizeof(HjdTableSet) * b->tsets.size();
    const size_t sz_qs = sizeof(HjdQuantSet) * b->qsets.size();
    const size_t sz_wk = sizeof(HjdEntropyWork) * b->work.size();
    const size_t sz_sg = sizeof(HjdEntropySeg) * b->segs.size();
    const size_t sz_s2 = sizeof(HjdSsSeg) * b->sssegs.size();
    const size_t sz_mc = sizeof(uint32_t) * b->mcu_cta.size();
    const size_t sz_sl = sizeof(HjdScanSlice) * b->slices.size();
    const size_t sz_is = sizeof(uint32_t) * b->host_istart.size();
    const size_t sz_ss = sizeof(HjdSsImage) * b->ss.size();
    const size_t sz_sw = sizeof(HjdSsWork) * b->sswork.size();
    const size_t sz_sd = sizeof(HjdScanDesc) * b->scans.size();
    const size_t sz_mw = sizeof(HjdMsWork) * b->mswork.size();
    const size_t sz_mst = sizeof(uint32_t) * b->ms_starts.size();
    const size_t sz_mt = sizeof(HjdHuffTable) * b->ms_tabs.size();
    if (sz_sd) {
        CU(b->d_scans.ensure(sz_sd));
        CU(b->d_mswork.ensure(sz_mw + 16));
        CU(b->d_msstarts.ensure(sz_mst + 16));
        CU(b->d_mstabs.ensure(sz_mt + 16));
    }
    size_t o_imgs = 0, o_ts = align_up(o_imgs + sz_imgs, 256), o_qs = align_up(o_ts + sz_ts, 256),
           o_wk = align_up(o_qs + sz_qs, 256), o_is = align_up(o_wk + sz_wk, 256),
           o_ss = align_up(o_is + sz_is, 256), o_sw = align_up(o_ss + sz_ss, 256),
           o_sg = align_up(o_sw + sz_sw, 256), o_s2 = align_up(o_sg + sz_sg, 256), o_mc = align_up(o_s2 + sz_s2, 256), o_sl = align_up(o_mc + sz_mc, 256),
           o_sd = align_up(o_sl + sz_sl, 256), o_mw = align_up(o_sd + sz_sd, 256), o_mst = align_up(o_mw + sz_mw, 256),
           o_mt = align_up(o_mst + sz_mst, 256), tot = o_mt + sz_mt;
    CU(b->h_meta.ensure(tot + 256));
    uint8_t* hm = (uint8_t*)b->h_meta.p;
    memcpy(hm + o_imgs, b->imgs.data(), sz_imgs);
    if (sz_ts) memcpy(hm + o_ts, b->tsets.data(), sz_ts);
    if (sz_qs) memcpy(hm + o_qs, b->qsets.data(), sz_qs);
    if (sz_wk) memcpy(hm + o_wk, b->work.data(), sz_wk);
    if (sz_sg) memcpy(hm + o_sg, b->segs.data(), sz_sg);
    if (sz_s2) memcpy(hm + o_s2, b->sssegs.data(), sz_s2);
    if (sz_mc) memcpy(hm + o_mc, b->mcu_cta.data(), sz_mc);
    if (sz_sl) memcpy(hm + o_sl, b->slices.data(), sz_sl);
    if (sz_is) memcpy(hm + o_is, b->host_istart.data(), sz_is);
    if (sz_ss) memcpy(hm + o_ss, b->ss.data(), sz_ss);
    if (sz_sw) memcpy(hm + o_sw, b->sswork.data(), sz_sw);
    if (sz_sd) {
        memcpy(hm + o_sd, b->scans.data(), sz_sd);
        memcpy(hm + o_mw, b->mswork.data(), sz_mw);
        memcpy(hm + o_mst, b->ms_starts.data(), sz_mst);
        memcpy(hm + o_mt, b->ms_tabs.data(), sz_mt);
        CU(cudaMemcpyAsync(b->d_scans.p, hm + o_sd, sz_sd, cudaMemcpyHostToDevice, b->stream));
        CU(cudaMemcpyAsync(b->d_mswork.p, hm + o_mw, sz_mw, cudaMemcpyHostToDevice, b->stream));
        CU(cudaMemcpyAsync(b->d_msstarts.p, hm + o_mst, sz_mst, cudaMemcpyHostToDevice, b->stream));
        CU(cudaMemcpyAsync(b->d_mstabs.p, hm + o_mt, sz_mt, cudaMemcpyHostToDevice, b->stream));
    }
    if (sz_imgs) CU(cudaMemcpyAsync(b->d_imgs.p, hm + o_imgs, sz_imgs, cudaMemcpyHostToDevice, b->stream));
    if (sz_ts) CU(cudaMemcpyAsync(b->d_tsets.p, hm + o_ts, sz_ts, cudaMemcpyHostToDevice, b->stream));
    if (sz_qs) CU(cudaMemcpyAsync(b->d_qsets.p, hm + o_qs, sz_qs, cudaMemcpyHostToDevice, b->stream));
    if (sz_wk) CU(cudaMemcpyAsync(b->d_work.p, hm + o_wk, sz_wk, cudaMemcpyHostToDevice, b->stream));
    if (sz_sg) CU(cudaMemcpyAsync(b->d_segs.p, hm + o_sg, sz_sg, cudaMemcpyHostToDevice, b->stream));
    if (sz_s2) CU(cudaMemcpyAsync(b->d_sssegs.p, hm + o_s2, sz_s2, cudaMemcpyHostToDevice, b->stream));
    if (sz_mc) CU(cudaMemcpyAsync(b->d_mcucta.p, hm + o_mc, sz_mc, cudaMemcpyHostToDevice, b->stream));
    if (sz_sl) CU(cudaMemcpyAsync(b->d_slices.p, hm + o_sl, sz_sl, cudaMemcpyHostToDevice, b->stream));
    if (sz_is) CU(cudaMemcpyAsync(b->d_istart.p, hm + o_is, sz_is, cudaMemcpyHostToDevice, b->stream));
    if (sz_ss) CU(cudaMemcpyAsync(b->d_ss.p, hm + o_ss, sz_ss, cudaMemcpyHostToDevice, b->stream));
    if (sz_sw) CU(cudaMemcpyAsync(b->d_sswork.p, hm + o_sw, sz_sw, cudaMemcpyHostToDevice, b->stream));
    CU(cudaMemsetAsync(b->d_status.p, 0, sizeof(int32_t) * (size_t)(n + 1), b->stream));

    b->uploaded = true;
    return HJD_OK;
}

// Host -> device copy of the files of images [img0, img1) (one copy for arena uploads).
static int copy_files(hjd_batch* b, const Chunk& c, cudaStream_t st)
{
    if (c.arena_hi <= c.arena_lo) return HJD_OK;
    if (b->contig_src) {
        CU(cudaMemcpyAsync((uint8_t*)b->d_arena.p + c.arena_lo, b->contig_src + c.arena_lo, c.arena_hi - c.arena_lo,
                           cudaMemcpyHostToDevice, st));
    } else {
        for (int i = c.img0; i < c.img1; i++) {
            const FileRef& f = b->files[i];
            if (f.ptr && f.size > 0)
                CU(cudaMemcpyAsync((uint8_t*)b->d_arena.p + f.dev_off, f.ptr, (size_t)f.size, cudaMemcpyHostToDevice, st));
        }
    }
    return HJD_OK;
}

static int prepare_separate(hjd_batch* b, const uint8_t* const* bufs, const int64_t* sizes, int n, bool chunked)
{
    b->files.assign((size_t)n, FileRef{nullptr, 0, 0});
    uint64_t off = 0;
    for (int i = 0; i < n; i++) {
        b->files[i] = FileRef{bufs[i], sizes[i], off};
        off += align_up(sizes[i] > 0 ? (uint64_t)sizes[i] : 0, 16);
    }
    b->arena_bytes = off;
    b->contig_src = nullptr;
    return upload_common(b, chunked);
}

static int prepare_arena(hjd_batch* b, const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n,
                         bool chunked)
{
    b->files.assign((size_t)n, FileRef{nullptr, 0, 0});
    int64_t lo = n ? offsets[0] : 0, hi = 0;
    for (int i = 0; i < n; i++) {
        if (offsets[i] < 0 || sizes[i] < 0) return fail(HJD_ERR_ARG, "hjd_batch_upload_arena", "negative offset/size");
        if (i && offsets[i] < offsets[i - 1]) return fail(HJD_ERR_ARG, "hjd_batch_upload_arena", "offsets must be ascending");
        if (offsets[i] < lo) lo = offsets[i];
        if (offsets[i] + sizes[i] > hi) hi = offsets[i] + sizes[i];
    }
    const int64_t lo_al = lo & ~(int64_t)15;      // keep the 16-byte phase of every file
    for (int i = 0; i < n; i++) b->files[i] = FileRef{arena + offsets[i], sizes[i], (uint64_t)(offsets[i] - lo_al)};
    b->arena_bytes = n ? (uint64_t)(hi - lo_al) : 0;
    b->contig_src = n ? arena + lo_al : nullptr;
    return upload_common(b, chunked);
}

extern "C" int hjd_batch_upload(hjd_batch* b, const uint8_t* const* bufs, const int64_t* sizes, int n)
{
    if (!b || !bufs || !sizes || n < 0) return fail(HJD_ERR_ARG, "hjd_batch_upload", "bad arguments");
    int rc = prepare_separate(b, bufs, sizes, n, b->overlap > 1);
    if (rc) return rc;
    for (const Chunk& c : b->chunks) { rc = copy_files(b, c, b->stream); if (rc) return rc; }
    return HJD_OK;
}

extern "C" int hjd_batch_upload_arena(hjd_batch* b, const uint8_t* arena, const int64_t* offsets,
                                      const int64_t* sizes, int n)
{
    if (!b || !arena || !offsets || !sizes || n < 0) return fail(HJD_ERR_ARG, "hjd_batch_upload_arena", "bad arguments");
    int rc = prepare_arena(b, arena, offsets, sizes, n, b->overlap > 1);
    if (rc) return rc;
    for (const Chunk& c : b->chunks) { rc = copy_files(b, c, b->stream); if (rc) return rc; }
    return HJD_OK;
}

extern "C" int hjd_batch_set_overlap(hjd_batch* b, int on)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_set_overlap", "null batch");
    b->overlap = on < 0 ? 0 : on;     // 0 serial, 1 default chunking, > 1: target blocks per chunk; next upload
    return HJD_OK;
}

extern "C" int hjd_batch_set_selfsync_range(hjd_batch* b, int range)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_set_selfsync_range", "null batch");
    if (range < 0 || range > HJD_SS_FIX_MAXR || (range & 31))
        return fail(HJD_ERR_ARG, "hjd_batch_set_selfsync_range", "range must be 0 or a multiple of 32 up to HJD_SS_FIX_MAXR");
    b->ss_range_req = (uint32_t)range;
    return HJD_OK;
}

// Kernel 1b for the restart-free images of one chunk (see selfsync.cu).  Everything is enqueued on `st`; the
// synchronisation rounds terminate on the device, so the host never waits here.
static int run_selfsync(hjd_batch* b, const Chunk& c, size_t chunk_index, cudaStream_t st)
{
    if (c.ss1 <= c.ss0) return HJD_OK;
    const uint8_t* arena = (const uint8_t*)b->d_arena.p;
    const HjdImageDesc* imgs = (const HjdImageDesc*)b->d_imgs.p;
    const HjdTableSet* tsets = (const HjdTableSet*)b->d_tsets.p;
    const HjdSsImage* ss = (const HjdSsImage*)b->d_ss.p;
    const HjdSsWork* work = (const HjdSsWork*)b->d_sswork.p + c.sw0;
    const HjdSsWork* work_fix = (const HjdSsWork*)b->d_sswork.p + c.sf0;
    const int n_work = (int)(c.sw1 - c.sw0), n_work_fix = (int)(c.sf1 - c.sf0);
    const HjdSsSeg* segs = (const HjdSsSeg*)b->d_sssegs.p;
    uint8_t* dst = (uint8_t*)b->d_destuff.p;
    uint32_t* dlen = (uint32_t*)b->d_dlen.p;
    uint64_t* E = (uint64_t*)b->d_ssE0.p;
    uint64_t* X = (uint64_t*)b->d_ssX.p;
    uint32_t* tmp = (uint32_t*)b->d_scantmp.p + chunk_index * b->ss_tmp_stride;
    uint32_t* ctl = (uint32_t*)b->d_flag.p + 4 * chunk_index;    // barrier count, last round with work, rounds run, item counter
    // [4][n_subs] (+ sentinel) counters of this chunk: starts, DC sums Y / Cb / Cr.  The kernels index them with
    // batch-wide sub-sequence numbers, hence the pointer that is shifted back by the chunk's first one.
    const uint32_t N = c.n_subs;
    uint32_t* cnt_region = (uint32_t*)b->d_ssnb.p + 4 * (size_t)c.sub0;
    uint32_t* cnt = cnt_region - c.sub0;

    CU(cudaMemsetAsync(ctl, 0, 4 * sizeof(uint32_t), st));
    CU(cudaMemsetAsync(cnt_region + 4 * (size_t)N, 0, sizeof(uint32_t), st));
    CU(hjd_launch_destuff(arena, imgs, ss + c.ss0, (int)(c.ss1 - c.ss0), c.ck0, c.n_ck, (uint32_t*)b->d_counts.p, tmp,
                          dst, dlen + c.ss0, st));
    b->launches += 2 + (c.n_ck + 1 > 2048 ? 3 : 1);
    CU(hjd_launch_ss_spec(imgs, tsets, ss, work, segs, n_work, dst, dlen, N, E, X, cnt, st));
    // a chain of wrong entry states can cross one range per round at worst: ranges + a confirming round
    const uint32_t max_rounds = N / 32 + 8;
    CU(hjd_launch_ss_sync(imgs, tsets, ss, work_fix, segs, n_work_fix, dst, dlen, N, E, X, cnt, ctl, max_rounds,
                          b->max_sync_ctas, st));
    CU(hjd_scan_u32(cnt_region, 4 * N + 1, tmp, st));                             // the counters become their exclusive prefix
    CU(hjd_launch_ss_write(imgs, tsets, ss, work, segs, n_work, dst, dlen, N, X, cnt, (int16_t*)b->d_coef.p,
                           (int32_t*)b->d_status.p, st));
    CU(hjd_launch_ss_fill_tail(imgs, ss + c.ss0, (int)(c.ss1 - c.ss0), cnt, (int16_t*)b->d_coef.p, st));
    b->launches += 4 + (4 * N + 1 > 2048 ? 3 : 1);
    b->ss_ran = true;
    return HJD_OK;
}

// Which fused kernel decodes a chunk's MCUs.  The tensor-core kernel (csrc/mcu_tc.cuh) is the faster one where its 128-MCU
// units are full and an MCU has several blocks to pipeline: large colour images (config 2: 3.39 ms against 3.63 ms, and the
// same time at every quality where the CUDA-core kernel's depends on the coefficients: 3.42 against 3.83 ms at q95; config 4:
// 0.221 against 0.242 ms).  Batches of small images are faster on the CUDA-core kernel (8192 thumbnails: 0.92 ms against
// 2.3 ms: a unit's set-up and pipeline fill are not amortised over one or two steps).
static int mcu_variant(unsigned flags, uint64_t blocks, uint32_t n_mcus, uint32_t n_images)
{
    if (flags & HJD_FLAG_TENSOR_CORE_IDCT) return HJD_MCU_TENSOR_CORE;
    if (flags & HJD_FLAG_CUDA_CORE_IDCT) return HJD_MCU_CUDA_CORE;
    // at least three blocks per MCU, at least eight full units per image, at least one unit for every group of every SM's CTA
    return (blocks >= 3ull * n_mcus && (uint64_t)n_mcus >= 1024ull * n_images && n_mcus >= 148u * 4u * 128u) ? HJD_MCU_TENSOR_CORE : HJD_MCU_CUDA_CORE;
}

// Kernels of one chunk on one stream.  ev != nullptr: record stage boundaries (serial mode only).
static int launch_chunk(hjd_batch* b, const Chunk& c, size_t chunk_index, cudaStream_t st, cudaEvent_t* ev)
{
    const uint8_t* arena = (const uint8_t*)b->d_arena.p;
    const HjdImageDesc* imgs = (const HjdImageDesc*)b->d_imgs.p;
    int32_t* status = (int32_t*)b->d_status.p;
    const int n = c.img1 - c.img0;
    if (!(b->flags & HJD_FLAG_HOST_SCAN) && n > 0) {
        CU(hjd_launch_marker_scan(arena, imgs, (uint32_t*)b->d_istart.p, status, c.img0, n,
                                  (const HjdScanSlice*)b->d_slices.p + c.slice0, (int)(c.slice1 - c.slice0),
                                  (uint32_t*)b->d_slicecnt.p + c.slice0, st));
        b->launches += 1 + (c.slice1 > c.slice0 ? 2 : 0);
    }
    if (ev) CU(cudaEventRecord(ev[1], st));
    {
        int rc = run_selfsync(b, c, chunk_index, st);      // counted in the entropy stage
        if (rc) return rc;
    }
    if (c.work1 > c.work0) {
        CU(hjd_launch_entropy_restart(arena, imgs, (const HjdTableSet*)b->d_tsets.p, (const uint32_t*)b->d_istart.p,
                                      (const HjdEntropyWork*)b->d_work.p + c.work0, (const HjdEntropySeg*)b->d_segs.p,
                                      (int)(c.work1 - c.work0),
                                      b->max_tabs, (int16_t*)b->d_coef.p, status, st));
        b->launches += 1;
    }
    // multi-scan images: nothing else writes their blocks, and refinement scans read what the levels below left
    for (const auto& z : c.ms_zero)
        CU(cudaMemsetAsync((int16_t*)b->d_coef.p + z.first * 64, 0, z.second * 128, st));
    for (const auto& lv : c.ms_levels) {
        CU(hjd_launch_multiscan(arena, imgs, (const HjdScanDesc*)b->d_scans.p, (const HjdMsWork*)b->d_mswork.p + lv.first,
                                (int)(lv.second - lv.first), (const uint32_t*)b->d_msstarts.p,
                                (const HjdHuffTable*)b->d_mstabs.p, (int16_t*)b->d_coef.p, status, st));
        b->launches += 1;
    }
    if (ev) CU(cudaEventRecord(ev[2], st));
    if (scale_shift(b->flags)) {
        // reduced-size decode: its own kernel in place of the fused one, counted in the same stage
        if (c.blocks) {
            b->sc_chunks++;
            CU(hjd_launch_mcu_rgb_scaled((const int16_t*)b->d_coef.p, imgs + c.img0, (const HjdQuantSet*)b->d_qsets.p,
                                         (uint8_t*)b->d_rgb.p, (const uint32_t*)b->d_mcucta.p + c.img0, n,
                                         b->mcu_cta[c.img1] - b->mcu_cta[c.img0], c.max_mcus, scale_shift(b->flags), st));
            b->launches += 1;
        }
        if (ev) CU(cudaEventRecord(ev[3], st));
    } else if (!(b->flags & HJD_FLAG_KEEP_PLANES)) {
        // default: kernels 2+3 fused per MCU, planes never reach HBM
        if (c.blocks) {
            const uint32_t n_mcus_chunk = b->mcu_cta[c.img1] - b->mcu_cta[c.img0];
            const int variant = mcu_variant(b->flags, c.blocks, n_mcus_chunk, (uint32_t)n);
            if (variant == HJD_MCU_TENSOR_CORE) b->tc_chunks++; else b->cc_chunks++;
            CU(hjd_launch_mcu_rgb((const int16_t*)b->d_coef.p, imgs + c.img0, (const HjdQuantSet*)b->d_qsets.p,
                                  (uint8_t*)b->d_rgb.p, (const uint32_t*)b->d_mcucta.p + c.img0, n,
                                  b->mcu_cta[c.img1] - b->mcu_cta[c.img0], c.max_mcus, (b->flags & HJD_FLAG_BMP_OUT) != 0,
                                  variant, st));
            b->launches += 1;
        }
        if (ev) CU(cudaEventRecord(ev[3], st));
    } else {
        if (c.blocks) {
            CU(hjd_launch_idct_planes((const int16_t*)b->d_coef.p, imgs + c.img0, (const HjdQuantSet*)b->d_qsets.p,
                                      (uint8_t*)b->d_planes.p, n, c.max_blocks, st));
            b->launches += (n + 65534) / 65535;
        }
        if (ev) CU(cudaEventRecord(ev[3], st));
        if (c.blocks) {
            CU(hjd_launch_color((const uint8_t*)b->d_planes.p, imgs + c.img0, (uint8_t*)b->d_rgb.p, n, c.max_w, c.max_h, st));
            b->launches += (n + 65534) / 65535;
        }
    }
    return HJD_OK;
}

// All chunks: optional H2D of the files, kernels, optional D2H of the RGB region into rgb_host.
static int run_chunks(hjd_batch* b, bool h2d, uint8_t* rgb_host)
{
    cudaStream_t main = b->stream;
    b->launches = 0;
    b->tc_chunks = b->cc_chunks = b->sc_chunks = 0;
    b->ss_ran = false;
    if (b->any_parse_error && b->rgb_bytes) CU(cudaMemsetAsync(b->d_rgb.p, 0, b->rgb_bytes, main));
    CU(cudaEventRecord(b->ev[0], main));
    if (b->chunks.size() <= 1) {
        // serial: one stream, stage boundaries recorded
        if (b->chunks.empty()) {
            for (int k = 1; k <= 3; k++) CU(cudaEventRecord(b->ev[k], main));
        } else {
            const Chunk& c = b->chunks[0];
            if (h2d) { int rc = copy_files(b, c, main); if (rc) return rc; CU(cudaEventRecord(b->ev[0], main)); }
            int rc = launch_chunk(b, c, 0, main, b->ev);
            if (rc) return rc;
        }
        CU(cudaEventRecord(b->ev[4], main));
        if (rgb_host && b->rgb_bytes) CU(cudaMemcpyAsync(rgb_host, b->d_rgb.p, b->rgb_bytes, cudaMemcpyDeviceToHost, main));
        return HJD_OK;
    }
    for (int k = 1; k <= 3; k++) CU(cudaEventRecord(b->ev[k], main));     // no per-stage times when chunks overlap
    CU(cudaEventRecord(b->ev_fork, main));
    for (int s = 0; s < HJD_NSTREAMS; s++) CU(cudaStreamWaitEvent(b->aux[s], b->ev_fork, 0));
    // From here on work is in flight on the chunk streams: whatever fails below, they are joined back into
    // the main stream before returning, so that the next upload (which synchronises only the main
    // stream before it rewrites the slabs) cannot overtake them.
    int rc_all = HJD_OK;
    for (size_t k = 0; k < b->chunks.size() && rc_all == HJD_OK; k++) {
        const Chunk& c = b->chunks[k];
        cudaStream_t st = b->aux[k % HJD_NSTREAMS];
        if (h2d) rc_all = copy_files(b, c, st);
        if (rc_all == HJD_OK) rc_all = launch_chunk(b, c, k, st, nullptr);
        if (rc_all == HJD_OK && rgb_host && c.rgb_hi > c.rgb_lo) {
            cudaError_t e = cudaMemcpyAsync(rgb_host + c.rgb_lo, (const uint8_t*)b->d_rgb.p + c.rgb_lo, c.rgb_hi - c.rgb_lo,
                                            cudaMemcpyDeviceToHost, st);
            if (e != cudaSuccess) rc_all = fail(HJD_ERR_CUDA, "cudaMemcpyAsync (RGB chunk)", cudaGetErrorString(e));
        }
    }
    for (int s = 0; s < HJD_NSTREAMS; s++) {
        cudaError_t e = cudaEventRecord(b->ev_join[s], b->aux[s]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(main, b->ev_join[s], 0);
        if (e != cudaSuccess) {
            cudaStreamSynchronize(b->aux[s]);                    // last resort: wait here
            if (rc_all == HJD_OK) rc_all = fail(HJD_ERR_CUDA, "joining the chunk streams", cudaGetErrorString(e));
        }
    }
    if (rc_all != HJD_OK) return rc_all;
    CU(cudaEventRecord(b->ev[4], main));
    return HJD_OK;
}

extern "C" int hjd_batch_decode(hjd_batch* b)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_decode", "null batch");
    if (!b->uploaded) return fail(HJD_ERR_STATE, "hjd_batch_decode", "nothing uploaded");
    CU(cudaSetDevice(b->device));
    int rc = run_chunks(b, false, nullptr);
    if (rc) return rc;
    b->decoded = true;
    return HJD_OK;
}

extern "C" int hjd_batch_sync(hjd_batch* b)
{
    if (!b) return fail(HJD_ERR_ARG, "hjd_batch_sync", "null batch");
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    return HJD_OK;
}

extern "C" int hjd_batch_num_images(const hjd_batch* b) { return b ? (int)b->imgs.size() : 0; }
extern "C" int hjd_batch_idct_variant(const hjd_batch* b)
{
    if (!b || (b->flags & HJD_FLAG_KEEP_PLANES)) return 0;
    return (b->tc_chunks ? 1 : 0) | (b->cc_chunks ? 2 : 0) | (b->sc_chunks ? 4 : 0);
}
extern "C" int hjd_batch_selfsync_rounds(hjd_batch* b)
{
    // rounds the device-side loop ran in the last decode (working rounds + the one that confirmed); syncs
    if (!b || !b->ss_ran || !b->d_flag.p) return 0;
    std::vector<uint32_t> ctl(4 * b->chunks.size() + 4, 0);
    if (cudaSetDevice(b->device) != cudaSuccess || cudaStreamSynchronize(b->stream) != cudaSuccess ||
        cudaMemcpy(ctl.data(), b->d_flag.p, 4 * b->chunks.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return -1; }
    uint32_t most = 0;                                             // the chunk that needed the most rounds
    for (size_t k = 0; k < b->chunks.size(); k++)
        if (b->chunks[k].ss1 > b->chunks[k].ss0 && (ctl[4 * k + 2] & 0x7FFFFFFFu) > most) most = ctl[4 * k + 2] & 0x7FFFFFFFu;
    return (int)most;
}

extern "C" int hjd_batch_get_info(const hjd_batch* b, int i, hjd_image_info* o)
{
    if (!b || !o || i < 0 || i >= (int)b->imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_get_info", "bad arguments");
    const HjdImageDesc& d = b->imgs[i];
    memset(o, 0, sizeof *o);
    o->width = d.width; o->height = d.height; o->ncomp = d.ncomp; o->hf = d.hf; o->vf = d.vf;
    o->blocks_per_mcu = d.blocks_per_mcu; o->mcus_x = d.mcus_x; o->mcus_y = d.mcus_y;
    o->restart_interval = d.restart_interval; o->n_intervals = d.n_intervals; o->scan_bytes = d.scan_len;
    o->block_base = d.block_base; o->n_blocks = d.n_blocks; o->rgb_offset = d.rgb_off;
    o->y_offset = d.y_off; o->cb_offset = d.cb_off; o->cr_offset = d.cr_off;
    o->y_pitch = d.y_pitch; o->c_pitch = d.c_pitch; o->status = b->parse_status[i];
    if (b->ms_items[i]) o->n_intervals = b->ms_items[i];
    return HJD_OK;
}

extern "C" int hjd_batch_get_out_size(const hjd_batch* b, int i, uint32_t* w, uint32_t* h)
{
    if (!b || i < 0 || i >= (int)b->imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_get_out_size", "bad arguments");
    const HjdImageDesc& d = b->imgs[i];
    if (w) *w = scaled_dim(b->flags, d.width);
    if (h) *h = scaled_dim(b->flags, d.height);
    return HJD_OK;
}

extern "C" int hjd_batch_num_scans(const hjd_batch* b, int i)
{
    if (!b || i < 0 || i >= (int)b->imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_num_scans", "bad arguments");
    return (int)b->n_scans[i];
}

extern "C" int hjd_batch_get_status(hjd_batch* b, int32_t* status)
{
    if (!b || !status) return fail(HJD_ERR_ARG, "hjd_batch_get_status", "bad arguments");
    CU(cudaSetDevice(b->device));
    const size_t n = b->imgs.size();
    if (n == 0) return HJD_OK;
    CU(cudaMemcpyAsync(status, b->d_status.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    if (b->ss_ran) {       // the device-side synchronisation loop reports here if it ever hit its round limit
        std::vector<uint32_t> ctl(4 * b->chunks.size() + 4, 0);
        CU(cudaMemcpy(ctl.data(), b->d_flag.p, 4 * b->chunks.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        for (size_t k = 0; k < b->chunks.size(); k++)
            if (b->chunks[k].ss1 > b->chunks[k].ss0 && (ctl[4 * k + 2] & 0x80000000u))
                return fail(HJD_ERR_STATE, "self-synchronising decode", "did not converge");
    }
    for (size_t i = 0; i < n; i++) {
        if (b->parse_status[i] != 0) status[i] = b->parse_status[i];
        else if (b->host_restart_warn[i]) status[i] |= HJD_IMG_WARN_RESTART;
    }
    return HJD_OK;
}

extern "C" int hjd_batch_get_timings(hjd_batch* b, hjd_timings* t)
{
    if (!b || !t) return fail(HJD_ERR_ARG, "hjd_batch_get_timings", "bad arguments");
    if (!b->decoded) return fail(HJD_ERR_STATE, "hjd_batch_get_timings", "no decode yet");
    CU(cudaSetDevice(b->device));
    CU(cudaEventSynchronize(b->ev[4]));
    CU(cudaEventElapsedTime(&t->scan_ms, b->ev[0], b->ev[1]));
    CU(cudaEventElapsedTime(&t->entropy_ms, b->ev[1], b->ev[2]));
    CU(cudaEventElapsedTime(&t->idct_ms, b->ev[2], b->ev[3]));
    CU(cudaEventElapsedTime(&t->color_ms, b->ev[3], b->ev[4]));
    CU(cudaEventElapsedTime(&t->total_ms, b->ev[0], b->ev[4]));
    t->launches = b->launches;
    return HJD_OK;
}

extern "C" int hjd_batch_mark(hjd_batch* b, int slot)
{
    if (!b || slot < 0 || slot >= HJD_MARK_SLOTS) return fail(HJD_ERR_ARG, "hjd_batch_mark", "bad arguments");
    CU(cudaSetDevice(b->device));
    CU(cudaEventRecord(b->mark[slot], b->stream));
    return HJD_OK;
}

extern "C" float hjd_batch_elapsed_ms(hjd_batch* b, int slot_a, int slot_b)
{
    if (!b || slot_a < 0 || slot_a >= HJD_MARK_SLOTS || slot_b < 0 || slot_b >= HJD_MARK_SLOTS) { fail(HJD_ERR_ARG, "hjd_batch_elapsed_ms", "bad arguments"); return -1.f; }
    float ms = -1.f;
    if (cudaSetDevice(b->device) != cudaSuccess || cudaEventSynchronize(b->mark[slot_b]) != cudaSuccess ||
        cudaEventElapsedTime(&ms, b->mark[slot_a], b->mark[slot_b]) != cudaSuccess) {
        fail(HJD_ERR_CUDA, "hjd_batch_elapsed_ms", cudaGetErrorString(cudaGetLastError()));
        return -1.f;
    }
    return ms;
}

extern "C" uint64_t hjd_batch_rgb_bytes(const hjd_batch* b)   { return b ? b->rgb_bytes : 0; }
extern "C" uint64_t hjd_batch_coef_bytes(const hjd_batch* b)  { return b ? b->total_blocks * 128 : 0; }
extern "C" uint64_t hjd_batch_plane_bytes(const hjd_batch* b) { return b ? b->plane_bytes : 0; }
extern "C" uint64_t hjd_batch_scan_bytes(const hjd_batch* b)  { return b ? b->scan_bytes : 0; }
extern "C" uint64_t hjd_batch_pixels(const hjd_batch* b)      { return b ? b->pixels : 0; }
extern "C" void* hjd_batch_device_rgb(hjd_batch* b)    { return b ? b->d_rgb.p : nullptr; }
extern "C" void* hjd_batch_device_coef(hjd_batch* b)   { return b ? b->d_coef.p : nullptr; }
extern "C" void* hjd_batch_device_planes(hjd_batch* b) { return b ? b->d_planes.p : nullptr; }

static int download(hjd_batch* b, void* dst, const void* src, uint64_t bytes, const char* who)
{
    if (!b || !dst) return fail(HJD_ERR_ARG, who, "bad arguments");
    if (!b->decoded) return fail(HJD_ERR_STATE, who, "no decode yet");
    CU(cudaSetDevice(b->device));
    if (bytes) CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return HJD_OK;
}

extern "C" int hjd_batch_download_rgb(hjd_batch* b, uint8_t* dst)
{ return download(b, dst, b ? b->d_rgb.p : nullptr, b ? b->rgb_bytes : 0, "hjd_batch_download_rgb"); }

extern "C" int hjd_batch_download_image(hjd_batch* b, int i, uint8_t* dst)
{
    if (!b || i < 0 || i >= (int)b->imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_download_image", "bad arguments");
    if (b->flags & HJD_FLAG_BMP_OUT) return fail(HJD_ERR_STATE, "hjd_batch_download_image", "this batch writes BMP files (HJD_FLAG_BMP_OUT): use hjd_batch_download_bmp");
    const HjdImageDesc& d = b->imgs[i];
    return download(b, dst, (const uint8_t*)b->d_rgb.p + d.rgb_off, image_out_bytes(b->flags, d.width, d.height),
                    "hjd_batch_download_image");
}

extern "C" uint64_t hjd_batch_bmp_bytes(const hjd_batch* b, int i)
{
    if (!b || i < 0 || i >= (int)b->imgs.size() || !(b->flags & HJD_FLAG_BMP_OUT) || b->parse_status[i] != HJD_IMG_OK) return 0;
    const HjdImageDesc& d = b->imgs[i];
    return 54 + (uint64_t)((d.width * 3 + 3) & ~3u) * d.height;                  // openjpg.cpp:541
}

extern "C" int hjd_batch_download_bmp(hjd_batch* b, int i, uint8_t* dst)
{
    if (!b || i < 0 || i >= (int)b->imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_download_bmp", "bad arguments");
    if (!(b->flags & HJD_FLAG_BMP_OUT)) return fail(HJD_ERR_STATE, "hjd_batch_download_bmp", "batch was not created with HJD_FLAG_BMP_OUT");
    const HjdImageDesc& d = b->imgs[i];
    return download(b, dst, (const uint8_t*)b->d_rgb.p + d.rgb_off + 10, hjd_batch_bmp_bytes(b, i), "hjd_batch_download_bmp");
}

extern "C" int hjd_batch_download_coef(hjd_batch* b, int16_t* dst)
{ return download(b, dst, b ? b->d_coef.p : nullptr, b ? b->total_blocks * 128 : 0, "hjd_batch_download_coef"); }

extern "C" int hjd_batch_download_image_coef(hjd_batch* b, int i, int16_t* dst)
{
    if (!b || i < 0 || i >= (int)b->imgs.size()) return fail(HJD_ERR_ARG, "hjd_batch_download_image_coef", "bad arguments");
    const HjdImageDesc& d = b->imgs[i];
    return download(b, dst, (const uint8_t*)b->d_coef.p + d.block_base * 128, d.n_blocks * 128, "hjd_batch_download_image_coef");
}

extern "C" int hjd_batch_download_planes(hjd_batch* b, uint8_t* dst)
{
    if (b && !(b->flags & HJD_FLAG_KEEP_PLANES)) return fail(HJD_ERR_STATE, "hjd_batch_download_planes", "planes exist in HBM only with HJD_FLAG_KEEP_PLANES (the default kernels keep them in shared memory)");
    return download(b, dst, b ? b->d_planes.p : nullptr, b ? b->plane_bytes : 0, "hjd_batch_download_planes");
}

// ------------------------------------------------------------------------------------------
// host-buffer end-to-end path
// ------------------------------------------------------------------------------------------
extern "C" uint64_t hjd_out_slab_bytes(const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n, unsigned flags)
{
    uint64_t total = 0;
    if (!arena || !offsets || !sizes) return 0;
    HjdParsed ps;
    std::unique_ptr<HjdMultiParsed> mp;
    for (int i = 0; i < n; i++) {
        int st = hjd_parse_jpeg(arena + offsets[i], (size_t)sizes[i], &ps);
        if (st == HJD_IMG_ERR_UNSUPPORTED && (flags & HJD_FLAG_MULTI_SCAN)) {
            if (!mp) mp.reset(new HjdMultiParsed());
            st = hjd_parse_jpeg_multi(arena + offsets[i], (size_t)sizes[i], mp.get());
            ps = mp->frame;
        }
        if (st == HJD_IMG_OK) total += align_up(image_out_bytes(flags, ps.width, ps.height), 256);
    }
    return total;
}

extern "C" uint64_t hjd_rgb_slab_bytes(const uint8_t* arena, const int64_t* offsets, const int64_t* sizes, int n)
{ return hjd_out_slab_bytes(arena, offsets, sizes, n, 0); }

extern "C" int hjd_batch_decode_host(hjd_batch* b, const uint8_t* arena, const int64_t* offsets, const int64_t* sizes,
                                     int n, uint8_t* rgb_out, uint64_t rgb_capacity, uint64_t* rgb_offsets_out,
                                     int32_t* status_out, int chunk_images)
{
    if (!b || !arena || !offsets || !sizes || !rgb_out || n < 0 || chunk_images < 0) return fail(HJD_ERR_ARG, "hjd_batch_decode_host", "bad arguments");
    CU(cudaSetDevice(b->device));
    b->chunk_images = chunk_images;                               // 0: chunks planned from the block counts (see upload_common)
    int rc = prepare_arena(b, arena, offsets, sizes, n, true);    // parse + metadata; files not copied yet
    b->chunk_images = 0;
    if (rc) return rc;
    if (b->rgb_bytes > rgb_capacity) return fail(HJD_ERR_ARG, "hjd_batch_decode_host", "rgb_out too small");
    rc = run_chunks(b, true, rgb_out);                            // per chunk: H2D, kernels, D2H
    if (rc) return rc;
    b->decoded = true;
    if (rgb_offsets_out)
        for (int i = 0; i < n; i++) rgb_offsets_out[i] = b->imgs[i].rgb_off;
    if (status_out) { rc = hjd_batch_get_status(b, status_out); if (rc) return rc; }
    CU(cudaStreamSynchronize(b->stream));
    return HJD_OK;
}

// NUMA node of a GPU (from sysfs via its PCI address), -1 when the platform does not say.
static int device_numa_node(int device)
{
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* p = bus; *p; p++) if (*p >= 'A' && *p <= 'F') *p = (char)(*p - 'A' + 'a');
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* fp = fopen(path, "r");
    if (!fp) return -1;
    int node = -1;
    if (fscanf(fp, "%d", &node) != 1) node = -1;
    fclose(fp);
    return node;
}

extern "C" int hjd_device_numa_node(int device) { return device_numa_node(device); }

// Pinned host memory whose pages come from the NUMA node next to `device` (set_mempolicy(MPOL_PREFERRED)
// around the allocation: cudaHostAlloc faults the pages in on the calling thread).  The D2H copy of a
// decoded batch is the end-to-end bottleneck, and a buffer on the far socket halves it on two-socket
// hosts.  Falls back to plain hjd_host_alloc when the platform exposes no NUMA topology.
extern "C" void* hjd_host_alloc_near(int device, size_t bytes)
{
    const int node = device_numa_node(device);
    bool bound = false;
#ifdef SYS_set_mempolicy
    if (node >= 0 && node < 1024) {
        unsigned long mask[16];
        memset(mask, 0, sizeof mask);
        mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
        bound = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, (unsigned long)(sizeof mask * 8)) == 0;
    }
#endif
    void* p = hjd_host_alloc(bytes);
#ifdef SYS_set_mempolicy
    if (bound) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
#endif
    (void)bound;
    return p;
}

// Raw link probe: `reps` times, concurrently on two streams and with no kernel anywhere, h2d_bytes from
// host_in to the device and d2h_bytes from the device to host_out (both pinned).  *ms = wall time of the
// slower direction per repetition.  This is the ceiling hjd_batch_decode_host works against.
extern "C" int hjd_link_probe(int device, const void* host_in, size_t h2d_bytes, void* host_out, size_t d2h_bytes,
                              int reps, float* ms_h2d, float* ms_d2h)
{
    if (reps <= 0) return fail(HJD_ERR_ARG, "hjd_link_probe", "bad arguments");
    CU(cudaSetDevice(device));
    void *d_in = nullptr, *d_out = nullptr;
    cudaStream_t s[2] = {nullptr, nullptr};
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int rc = HJD_OK;
    auto cleanup = [&]() {
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        for (auto& q : s) if (q) cudaStreamDestroy(q);
        if (d_in) cudaFree(d_in);
        if (d_out) cudaFree(d_out);
    };
    cudaError_t e = cudaSuccess;
    if (h2d_bytes && host_in) e = cudaMalloc(&d_in, h2d_bytes);
    if (e == cudaSuccess && d2h_bytes && host_out) e = cudaMalloc(&d_out, d2h_bytes);
    for (int k = 0; k < 2 && e == cudaSuccess; k++) e = cudaStreamCreateWithFlags(&s[k], cudaStreamNonBlocking);
    for (int k = 0; k < 4 && e == cudaSuccess; k++) e = cudaEventCreate(&ev[k]);
    if (e == cudaSuccess && d_out) e = cudaMemset(d_out, 0x5a, d2h_bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) {
        cudaEventRecord(ev[0], s[0]); cudaEventRecord(ev[2], s[1]);
        for (int r = 0; r < reps; r++) {
            if (d_in) cudaMemcpyAsync(d_in, host_in, h2d_bytes, cudaMemcpyHostToDevice, s[0]);
            if (d_out) cudaMemcpyAsync(host_out, d_out, d2h_bytes, cudaMemcpyDeviceToHost, s[1]);
        }
        cudaEventRecord(ev[1], s[0]); cudaEventRecord(ev[3], s[1]);
        e = cudaStreamSynchronize(s[0]);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s[1]);
        float a = 0.f, b = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&a, ev[0], ev[1]);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&b, ev[2], ev[3]);
        if (ms_h2d) *ms_h2d = a / (float)reps;
        if (ms_d2h) *ms_d2h = b / (float)reps;
    }
    if (e != cudaSuccess) rc = fail(HJD_ERR_CUDA, "hjd_link_probe", cudaGetErrorString(e));
    cleanup();
    return rc;
}

extern "C" void* hjd_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); fail(HJD_ERR_NOMEM, "cudaHostAlloc"); return nullptr; }
    return p;
}
extern "C" void hjd_host_free(void* p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------
// reference-shaped single-image calls
// ------------------------------------------------------------------------------------------
struct DefaultBatch {
    hjd_batch* b[2] = {nullptr, nullptr};      // [0] RGB out (DecodeJpgFileData), [1] BMP out (ConvertJpgFile)
    int device[2] = {-1, -1};
    ~DefaultBatch() { for (int k = 0; k < 2; k++) if (b[k]) hjd_batch_destroy(b[k]); }
};
static thread_local DefaultBatch g_default;
static std::atomic<int> g_default_device(0);

extern "C" int hjd_set_default_device(int device)
{
    if (device < 0 || device >= hjd_device_count()) return fail(HJD_ERR_ARG, "hjd_set_default_device", "bad device index");
    g_default_device.store(device);
    return HJD_OK;
}

// The lazily created per-thread batch behind the single-image calls, on the process-wide default device.
static hjd_batch* default_batch(bool bmp)
{
    const int k = bmp ? 1 : 0, dev = g_default_device.load();
    if (g_default.b[k] && g_default.device[k] != dev) { hjd_batch_destroy(g_default.b[k]); g_default.b[k] = nullptr; }
    if (!g_default.b[k]) { g_default.b[k] = hjd_batch_create(dev, bmp ? HJD_FLAG_BMP_OUT : 0); g_default.device[k] = dev; }
    return g_default.b[k];
}

extern "C" void hjd_free(void* p) { free(p); }

extern "C" int hjd_get_image_size(const uint8_t* buf, int size, unsigned* width, unsigned* height)
{
    HjdParsed ps;
    if (!buf || size <= 0 || hjd_parse_jpeg(buf, (size_t)size, &ps) != HJD_IMG_OK) { fail(HJD_ERR_ARG, "hjd_get_image_size", "not a decodable baseline JPEG"); return 0; }
    if (width) *width = ps.width;
    if (height) *height = ps.height;
    return 1;
}

static void fill_info_from_parse(const HjdParsed& ps, hjd_image_info* o)
{
    memset(o, 0, sizeof *o);
    o->status = ps.status;
    if (ps.status != HJD_IMG_OK) return;
    o->width = ps.width; o->height = ps.height; o->ncomp = (uint8_t)ps.ncomp; o->hf = (uint8_t)ps.hf; o->vf = (uint8_t)ps.vf;
    o->blocks_per_mcu = (uint8_t)(ps.ncomp == 3 ? ps.hf * ps.vf + 2 : 1);
    o->mcus_x = (ps.width + 8 * ps.hf - 1) / (8 * ps.hf);
    o->mcus_y = (ps.height + 8 * ps.vf - 1) / (8 * ps.vf);
    o->restart_interval = ps.restart_interval;
    const uint32_t n_mcus = o->mcus_x * o->mcus_y;
    o->n_intervals = ps.restart_interval ? (n_mcus + ps.restart_interval - 1) / ps.restart_interval : 1;
    o->scan_bytes = (uint32_t)ps.scan_len;
    o->n_blocks = (uint64_t)n_mcus * o->blocks_per_mcu;
}

extern "C" int hjd_probe_jpeg(const uint8_t* buf, int64_t size, hjd_image_info* out)
{
    HjdParsed ps;
    const int st = (buf && size > 0) ? hjd_parse_jpeg(buf, (size_t)size, &ps) : HJD_IMG_ERR_NOT_JPEG;
    if (buf && size > 0 && st == HJD_IMG_OK) {
        HjdTableSet ts;
        ps.status = hjd_build_table_set(ps, &ts);                  // an over-subscribed DHT is a per-image error too
    } else ps.status = st;
    if (out) fill_info_from_parse(ps, out);
    return ps.status;
}

// Multi-scan parse plus every table build: the status a batch with HJD_FLAG_MULTI_SCAN reports for the file.
static int probe_multi(const uint8_t* buf, int64_t size, HjdMultiParsed* mp)
{
    int st = hjd_parse_jpeg_multi(buf, (size_t)size, mp);
    if (st == HJD_IMG_OK && mp->frame.scan_len > 0xFFFFFF00ull) st = HJD_IMG_ERR_UNSUPPORTED;
    HjdHuffTable t;
    for (size_t k = 0; st == HJD_IMG_OK && k < mp->scans.size(); k++) {
        const HjdScanParsed& s = mp->scans[k];
        for (int c = 0; c < s.ncomp; c++) {
            if (s.dc[c].present && !hjd_build_huff_table(s.dc[c], false, &t)) st = HJD_IMG_ERR_BAD_TABLE;
            if (s.ac[c].present && !(s.kind == HJD_SCAN_SEQ ? hjd_build_huff_table(s.ac[c], true, &t) : hjd_build_huff_table_raw(s.ac[c], &t)))
                st = HJD_IMG_ERR_BAD_TABLE;
        }
    }
    return mp->frame.status = st;
}

extern "C" int hjd_probe_jpeg_flags(const uint8_t* buf, int64_t size, unsigned flags, hjd_image_info* out)
{
    const int st = hjd_probe_jpeg(buf, size, out);
    if (st != HJD_IMG_ERR_UNSUPPORTED || !(flags & HJD_FLAG_MULTI_SCAN)) return st;
    std::unique_ptr<HjdMultiParsed> mp(new HjdMultiParsed());
    probe_multi(buf, size, mp.get());
    const HjdParsed& f = mp->frame;
    if (out) {
        fill_info_from_parse(f, out);
        if (f.status == HJD_IMG_OK) {
            out->n_intervals = 0;
            for (const HjdScanParsed& s : mp->scans) {
                if (scale_shift(flags) == 3 && s.ss > 0) continue;      // not read at 1/8 (see ms_add_image)
                uint32_t mx, my;
                hjd_scan_grid(f, s, &mx, &my);
                const uint64_t want = s.restart_interval ? ((uint64_t)mx * my + s.restart_interval - 1) / s.restart_interval : 1;
                out->n_intervals += (uint32_t)(want < s.n_starts ? want : s.n_starts);
            }
        }
    }
    return f.status;
}

extern "C" int hjd_probe_jpeg_scans(const uint8_t* buf, int64_t size, hjd_scan_info* out, int max)
{
    if (max < 0 || (max > 0 && !out)) return fail(HJD_ERR_ARG, "hjd_probe_jpeg_scans", "bad arguments");
    hjd_image_info info;
    const int st = hjd_probe_jpeg(buf, size, &info);
    if (st == HJD_IMG_OK) {                       // one interleaved sequential scan
        if (max > 0) {
            memset(out, 0, sizeof *out);
            out->ncomp = info.ncomp;
            for (int c = 0; c < info.ncomp; c++) out->comp[c] = (uint8_t)c;
            out->se = 63;
            out->restart_interval = info.restart_interval;
            out->bytes = info.scan_bytes;
        }
        return 1;
    }
    if (st != HJD_IMG_ERR_UNSUPPORTED) return st;
    std::unique_ptr<HjdMultiParsed> mp(new HjdMultiParsed());
    const int ms = probe_multi(buf, size, mp.get());
    if (ms != HJD_IMG_OK) return ms;
    for (int k = 0; k < (int)mp->scans.size() && k < max; k++) {
        const HjdScanParsed& s = mp->scans[(size_t)k];
        hjd_scan_info& o = out[k];
        memset(&o, 0, sizeof o);
        o.ncomp = (uint8_t)s.ncomp;
        for (int c = 0; c < s.ncomp; c++) o.comp[c] = (uint8_t)s.comp[c];
        o.ss = (uint8_t)s.ss; o.se = (uint8_t)s.se; o.ah = (uint8_t)s.ah; o.al = (uint8_t)s.al;
        o.level = (uint8_t)(s.level < 255 ? s.level : 255);
        o.restart_interval = s.restart_interval;
        o.bytes = (uint32_t)s.len;
    }
    return (int)mp->scans.size();
}

extern "C" uint32_t hjd_huff_lookup_probe(const uint8_t bits[16], const uint8_t* vals, int nvals, int is_ac, uint32_t peek16)
{
    static thread_local HjdHuffTable tab;
    static thread_local HjdRawHuff cached;
    static thread_local int cached_ac = -1;
    HjdRawHuff raw;
    memset(&raw, 0, sizeof raw);
    if (!bits || !vals || nvals < 0 || nvals > 256) return 0xFFFFFFFFu;
    memcpy(raw.bits, bits, 16);
    memcpy(raw.vals, vals, (size_t)nvals);
    raw.nvals = nvals;
    raw.present = 1;
    if (cached_ac != is_ac || memcmp(&cached, &raw, sizeof raw) != 0) {
        cached_ac = -1;
        if (!hjd_build_huff_table(raw, is_ac != 0, &tab)) return 0xFFFFFFFFu;
        cached = raw;
        cached_ac = is_ac;
    }
    return hjd_host_huff_lookup(&tab, peek16);
}

// One image through a default batch; the result (RGB24, or the BMP file) is downloaded into memory from
// alloc(bytes).  The staging is the batch's own pinned buffer: one asynchronous copy, one host copy.
static int decode_one(bool bmp, const uint8_t* buf, int size, void* (*alloc)(size_t), uint8_t** out_ptr, size_t* out_bytes,
                      unsigned* width, unsigned* height, const char* who)
{
    if (!buf || size <= 0 || !out_ptr || !alloc) { fail(HJD_ERR_ARG, who, "bad arguments"); return 0; }
    *out_ptr = nullptr;
    hjd_batch* b = default_batch(bmp);
    if (!b) return 0;
    const uint8_t* bufs[1] = {buf};
    const int64_t sizes[1] = {size};
    if (hjd_batch_upload(b, bufs, sizes, 1) != HJD_OK) return 0;
    if (b->parse_status[0] != HJD_IMG_OK) { fail(HJD_ERR_ARG, who, "unsupported or corrupt JPEG"); return 0; }
    if (hjd_batch_decode(b) != HJD_OK) return 0;
    const HjdImageDesc& d = b->imgs[0];
    const size_t bytes = bmp ? (size_t)hjd_batch_bmp_bytes(b, 0) : (size_t)d.width * d.height * 3;
    if (cudaSetDevice(b->device) != cudaSuccess || b->h_out.ensure(bytes + 16) != cudaSuccess) { cudaGetLastError(); fail(HJD_ERR_NOMEM, who, "pinned staging buffer"); return 0; }
    if (cudaMemcpyAsync(b->h_out.p, (const uint8_t*)b->d_rgb.p + d.rgb_off + (bmp ? 10 : 0), bytes, cudaMemcpyDeviceToHost, b->stream) != cudaSuccess ||
        cudaStreamSynchronize(b->stream) != cudaSuccess) { fail(HJD_ERR_CUDA, who, cudaGetErrorString(cudaGetLastError())); return 0; }
    uint8_t* out = (uint8_t*)alloc(bytes ? bytes : 1);
    if (!out) { fail(HJD_ERR_NOMEM, who, "allocation failed"); return 0; }
    memcpy(out, b->h_out.p, bytes);
    *out_ptr = out;
    if (out_bytes) *out_bytes = bytes;
    if (width) *width = d.width;
    if (height) *height = d.height;
    return 1;
}

extern "C" int hjd_decode_jpg_file_data_alloc(const uint8_t* buf, int size, void* (*alloc)(size_t), uint8_t** rgb,
                                              unsigned* width, unsigned* height)
{
    return decode_one(false, buf, size, alloc, rgb, nullptr, width, height, "hjd_decode_jpg_file_data");
}

extern "C" int hjd_decode_jpg_file_data(const uint8_t* buf, int size, uint8_t** rgb, unsigned* width, unsigned* height)
{
    return decode_one(false, buf, size, malloc, rgb, nullptr, width, height, "hjd_decode_jpg_file_data");
}

extern "C" size_t hjd_encode_bmp24(unsigned width, unsigned height, const uint8_t* rgb, uint8_t* out)
{
    // openjpg.cpp:504-570: 14+40 byte header, bottom-up, B G R, each row padded to a multiple of 4.
    const unsigned pad = (4 - (width * 3) % 4) % 4;
    const size_t total = (size_t)width * height * 3 + (size_t)height * pad + 54;
    if (!out) return total;
    memset(out, 0, 54);
    auto put32 = [&](int at, uint32_t v) { out[at] = v & 255; out[at + 1] = (v >> 8) & 255; out[at + 2] = (v >> 16) & 255; out[at + 3] = (v >> 24) & 255; };
    out[0] = 'B'; out[1] = 'M';
    put32(2, (uint32_t)total);
    put32(10, 54);
    put32(14, 40);
    put32(18, width);
    put32(22, height);
    out[26] = 1;
    out[28] = 24;
    uint8_t* o = out + 54;
    for (unsigned row = height; row-- > 0;) {
        const uint8_t* src = rgb + (size_t)row * width * 3;
        for (unsigned x = 0; x < width; x++) { o[0] = src[2]; o[1] = src[1]; o[2] = src[0]; o += 3; src += 3; }
        for (unsigned k = 0; k < pad; k++) *o++ = 0;
    }
    return total;
}

extern "C" int hjd_write_bmp24(const char* path, unsigned width, unsigned height, const uint8_t* rgb)
{
    if (!path || !rgb) { fail(HJD_ERR_ARG, "hjd_write_bmp24", "bad arguments"); return 0; }
    const size_t total = hjd_encode_bmp24(width, height, rgb, nullptr);
    uint8_t* tmp = (uint8_t*)malloc(total);
    if (!tmp) { fail(HJD_ERR_NOMEM, "malloc"); return 0; }
    hjd_encode_bmp24(width, height, rgb, tmp);
    FILE* fp = fopen(path, "wb");
    if (!fp) { free(tmp); fail(HJD_ERR_IO, "fopen", path); return 0; }
    const size_t w = fwrite(tmp, 1, total, fp);
    fclose(fp);
    free(tmp);
    if (w != total) { fail(HJD_ERR_IO, "fwrite", path); return 0; }
    return 1;
}

extern "C" int hjd_convert_jpg_file(const char* jpg_in, const char* bmp_out)
{
    // ConvertJpgFile, openjpg.cpp:593-684: returns 1 on success, 0 on failure.  The decode runs with
    // HJD_FLAG_BMP_OUT: what comes back from the GPU is the file WriteBMP24 would write.
    if (!jpg_in || !bmp_out) { fail(HJD_ERR_ARG, "hjd_convert_jpg_file", "bad arguments"); return 0; }
    FILE* fp = fopen(jpg_in, "rb");
    if (!fp) { fail(HJD_ERR_IO, "fopen", jpg_in); return 0; }          // openjpg.cpp:603-608
    fseek(fp, 0, SEEK_END);
    const long len = ftell(fp);
    fseek(fp, 0, SEEK_SET);
    if (len <= 0 || len > 0x7FFFFFFF) { fclose(fp); fail(HJD_ERR_IO, "empty or oversized file", jpg_in); return 0; }
    uint8_t* buf = (uint8_t*)malloc((size_t)len);
    if (!buf) { fclose(fp); fail(HJD_ERR_NOMEM, "malloc"); return 0; }
    const size_t got = fread(buf, 1, (size_t)len, fp);
    fclose(fp);
    uint8_t* bmp = nullptr;
    size_t bytes = 0;
    int ok = (got == (size_t)len) && decode_one(true, buf, (int)len, malloc, &bmp, &bytes, nullptr, nullptr, "hjd_convert_jpg_file");
    free(buf);
    if (!ok) return 0;
    fp = fopen(bmp_out, "wb");
    if (!fp) { free(bmp); fail(HJD_ERR_IO, "fopen", bmp_out); return 0; }
    ok = fwrite(bmp, 1, bytes, fp) == bytes;
    if (fclose(fp) != 0) ok = 0;
    free(bmp);
    if (!ok) fail(HJD_ERR_IO, "fwrite", bmp_out);
    return ok;
}
